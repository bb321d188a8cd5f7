#!/usr/bin/env python
"""bench.py — M-LOAM per-scan hot path on B200 (contract: see the task statement / DESIGN.md §Measurement).

A "step" is one pass of the hot path over one synthetic rig frame (the sweeps of all LiDARs of the configuration):
    FeatureExtract::extractCloud per LiDAR -> extrinsic + laser id merge -> downsampleCurrentScan -> scan2MapOptimization with
    GN re-association iterations (kNN + line/plane fit + residual/Jacobian + J^T J reduction + LM step each), plus — on keyframe
    steps — setInputCloud on the surf + corner submaps (upload + rebuild).
Workloads (BASELINE.json configs; --config overrides the default picked from --gpus):
    C2  1 LiDAR  64 x 2048, 1M-point submap, 10 GN iterations                    (default at --gpus 1)
    C3  2 LiDARs 64 x 2048, 2M-point submap, 12-DoF online extrinsic calibration (default at --gpus 2)
    C4  4 LiDARs (RV rig) 64 x 2048, 5M-point submap                              (default at --gpus 4; `--gpus 1 --config C4`
                                                                                  is the north star's ">= 50x on 4 x 64-ring LiDARs at 1 GPU")
    C5  8 LiDARs 128 x 2048, 10M-point submap, greedy good-feature selection 0.8  (default at --gpus 8)
The LiDARs are sharded over the GPUs (lidars / gpus per GPU, batched in one context each); the submap is replicated; the
packed normal equations are summed over the GPUs at every LM evaluation.

The submap only changes when the mapper saves a keyframe (lidar_mapper_keyframe.cpp:1101; DISTANCE_KEYFRAMES = 1 m =
every 10th frame at the trajectory's 1 m/s, 10 Hz): the GPU keeps it resident and rebuilds it on keyframe steps only
(`keyframe_every`); the reference — and therefore the CPU arm — rebuilds its kd-trees every frame (:433-434).

value       : LiDAR sweeps through the whole hot path per second, summed over GPUs, inputs resident in HBM.
e2e         : the same through the C-ABI call a user makes (mloam_frame) with HOST buffers (pinned): H2D of the sweeps every
              step, of both submaps on keyframe steps, D2H of the pose + solver state.
roofline    : k_match_knn (dominant) and the map build (the streaming kernel), algorithmic bytes / CUDA-event time.
cpu_baseline: the CPU restatement of the reference path (oracle/, kd-tree = the reference's own nanoflann from oracle/_ref)
              on the same frames, reference threading.  --impl reference: that CPU path as the timed arm.
"""
from __future__ import annotations

import argparse
import importlib.util
import json
import math
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.dont_write_bytecode = True  # the tree may be read-only: no __pycache__ for the modules imported from it

METRIC = "scan_to_map_lidar_frames_per_sec"
KEYFRAME_EVERY = 10
CONFIGS = {
    "C2": dict(lidars=1, rings=64, horizon=2048, map_points=1_000_000, gn_iters=10, gf_method=0, gf_ratio=1.0, calib=False),
    "C3": dict(lidars=2, rings=64, horizon=2048, map_points=2_000_000, gn_iters=10, gf_method=0, gf_ratio=1.0, calib=True),
    "C4": dict(lidars=4, rings=64, horizon=2048, map_points=5_000_000, gn_iters=10, gf_method=0, gf_ratio=1.0, calib=False),
    "C5": dict(lidars=8, rings=128, horizon=2048, map_points=10_000_000, gn_iters=10, gf_method=3, gf_ratio=0.8, calib=False),
}
DEFAULT_CONFIG = {1: "C2", 2: "C3", 4: "C4", 8: "C5"}
SOLVE_STATS = ("ran", "n_surf", "n_corner", "lm_iterations", "degenerate", "termination", "final_cost", "eig", "H", "n_surf_in", "n_corner_in")
KNN_BYTES_PER_FEATURE = 16 + 5 * 16 + 5 * 4   # k_match_knn: query float4 + 5 neighbour float4 + 5 neighbour positions
MAP_BYTES_PER_POINT = 40                     # map build: 16 read + 16 sorted write + 8 key/rank (SURVEY.md §8d)


def load_mloam():
    spec = importlib.util.spec_from_file_location("mloam_b200", os.path.join(ROOT, "m-loam_b200", "__init__.py"))
    mod = importlib.util.module_from_spec(spec)
    sys.modules["mloam_b200"] = mod
    spec.loader.exec_module(mod)
    return mod


def lidar_extrinsic(syn, rank: int, n: int):
    """Extrinsic of LiDAR `rank` of an n-LiDAR rig (kept for tests/multi_gpu_check.py)."""
    return None if rank == 0 else syn.rig_extrinsics(max(n, 5) if n > 4 else n)[rank]


def _oracle_fn(name):
    def f(*a, **k):  # only reached when tests/golden/submap_keyframes_filtered.npz is missing (it is committed)
        import oracle_lib as orc
        return getattr(orc, name)(*a, **k)
    return f


def make_submap(syn, scene, n_total: int, kind: str):
    if kind == "uniform":
        s, c = syn.make_submap(scene, n_total)
        return s, c, {"kind": "uniform: area / length-uniform samples of the scene geometry, 1 cm jitter"}
    s, c, info = syn.make_submap_keyframes(scene, n_total, _oracle_fn("extract_cloud"), _oracle_fn("voxel_grid"))
    info["kind"] = ("keyframes (SURVEY.md 8d): 30 ray-cast keyframes -> extractCloud -> VoxelGrid 0.2 / 0.4 -> re-sampled with 1 cm jitter to the "
                    "configuration's size")
    return s, c, info


def make_workload(syn, cfg: dict, n_gpus: int, rank: int, n_frames: int, map_kind: str = "keyframes", all_groups: bool = False):
    """Per-rank workload.  The LiDARs of the rig are split into n_gpus consecutive groups; rank r gets group r."""
    L = cfg["lidars"]
    scene = syn.make_scene()
    traj = syn.trajectory(n_frames + 2)
    surf_map, corner_map, map_info = make_submap(syn, scene, cfg["map_points"], map_kind)
    ext_all = syn.rig_extrinsics(L)
    per = max(1, L // n_gpus)
    groups = [list(range(g * per, min(L, (g + 1) * per))) for g in range(n_gpus)]
    rng = np.random.Generator(np.random.PCG64(1234))
    frames = []
    for k in range(n_frames):
        truth = traj[k + 1]
        init = syn.perturb_pose(truth, rng)  # BASE pose guess, identical on every rank (shared state of the summed LM)
        fr = dict(init=init, truth=truth, groups={})
        for g, ids in enumerate(groups):
            if not ids or (g != rank and not all_groups):
                continue
            clouds, starts, ends, base = [], [], [], 0
            for l in ids:
                c, ss, se = syn.make_sweep(scene, truth, cfg["rings"], cfg["horizon"], seed=100 + k, lidar_id=l, ext=ext_all[l])
                clouds.append(c), starts.append(ss + base), ends.append(se + base)
                base += c.shape[0]
            fr["groups"][g] = dict(cloud=np.ascontiguousarray(np.concatenate(clouds)), ss=np.concatenate(starts).astype(np.int32),
                                   se=np.concatenate(ends).astype(np.int32), ext=ext_all[ids])
        frames.append(fr)
    return dict(surf_map=surf_map, corner_map=corner_map, map_info=map_info, frames=frames, groups=groups, ext_all=ext_all)


class ClockSampler:
    """SM clock / throttle reasons DURING the timed region (B200_PROFILING.md's clocks line), sampled in-process
    through NVML every 10 ms — an `nvidia-smi -lms` child was seen to stall kernel submission for milliseconds at a
    time on these hosts, which is not what a 1.5 ms step should be measured next to.  Falls back to that child when
    NVML is not importable."""

    REASONS = (("hw_slowdown", "nvmlClocksEventReasonHwSlowdown"), ("hw_thermal_slowdown", "nvmlClocksEventReasonHwThermalSlowdown"),
               ("sw_thermal_slowdown", "nvmlClocksEventReasonSwThermalSlowdown"), ("sw_power_cap", "nvmlClocksEventReasonSwPowerCap"))

    def __init__(self, index: int):
        self.index, self.rows, self.proc, self.nvml, self.stop_flag = index, [], None, None, False
        self.t_begin = 0.0

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[self.index]) if vis and vis.split(",")[self.index].strip().isdigit() else self.index
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_sm = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
            self.t = threading.Thread(target=self._poll_nvml, daemon=True)
            self.t.start()
            return
        except Exception:
            self.nvml = None
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read_smi, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _poll_nvml(self):
        n = self.nvml
        while not self.stop_flag:
            try:
                sm = float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM))
                mask = int(n.nvmlDeviceGetCurrentClocksEventReasons(self.handle))
                active = [name for name, attr in self.REASONS if mask & int(getattr(n, attr))]
                self.rows.append((time.perf_counter(), sm, self.max_sm, active))
            except Exception:
                pass
            time.sleep(0.01)

    def _read_smi(self):
        for line in self.proc.stdout:
            f = [x.strip() for x in line.strip().split(",")]
            if len(f) < 7:
                continue
            try:
                sm, mx = float(f[0]), float(f[1])
            except ValueError:
                continue
            active = [name for (name, _), v in zip(self.REASONS, f[3:7]) if v.lower().startswith("active")]
            self.rows.append((time.perf_counter(), sm, mx, active))

    def wait_first(self, timeout=15.0):
        t0 = time.perf_counter()
        while (self.nvml is not None or self.proc is not None) and not self.rows and time.perf_counter() - t0 < timeout:
            time.sleep(0.02)

    def mark(self):
        self.t_begin = time.perf_counter()

    def stop(self) -> dict:
        t_end = time.perf_counter()
        self.stop_flag = True
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                pass
        if self.nvml is None and self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no NVML / nvidia-smi"], "samples": 0}
        inside = [r for r in self.rows if self.t_begin <= r[0] <= t_end + 0.02]
        if not inside:  # timed region shorter than one sampling period: the closest samples taken under load
            inside = self.rows[-2:]
        sm = [r[1] for r in inside]
        mx = [r[2] for r in inside]
        reasons = sorted({x for r in inside for x in r[3]})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm), "source": "nvml" if self.nvml is not None else "nvidia-smi"}


def oracle_opts(orc, cfg):
    o = orc.default_opts()
    o[orc.O_MAX_OUTER], o[orc.O_MAX_INNER] = cfg["gn_iters"], 1
    o[orc.O_GF_METHOD], o[orc.O_GF_RATIO], o[orc.O_GF_SEED] = cfg["gf_method"], cfg["gf_ratio"], 0
    return o


def oracle_frame(orc, cfg, wl, fr, sharded: bool):
    """The oracle's pose for one rig frame.  sharded: features prepared per GPU group (merged down-sampling inside a group,
    good-feature selection per group) as the N-GPU run does; otherwise the reference's single merged list."""
    o = oracle_opts(orc, cfg)
    gids = sorted(fr["groups"])
    if not sharded or len(gids) == 1:
        g = fr["groups"][gids[0]] if len(gids) == 1 else None
        if g is None:  # merge all groups' raw sweeps into one rig frame
            clouds, ss, se, ext, base = [], [], [], [], 0
            for q in gids:
                G = fr["groups"][q]
                clouds.append(G["cloud"]), ss.append(G["ss"] + base), se.append(G["se"] + base), ext.append(G["ext"])
                base += G["cloud"].shape[0]
            g = dict(cloud=np.concatenate(clouds), ss=np.concatenate(ss).astype(np.int32), se=np.concatenate(se).astype(np.int32),
                     ext=np.concatenate(ext))
        return orc.frame_multi(g["cloud"], g["ss"], g["se"], g["ext"].shape[0], g["ext"], wl["surf_map"], wl["corner_map"], fr["init"], o)
    cs_all, sf_all = [], []
    for q in gids:
        G = fr["groups"][q]
        cs, sf = orc.prepare_multi(G["cloud"], G["ss"], G["se"], G["ext"].shape[0], G["ext"])
        cs_all.append(cs), sf_all.append(sf)
    if cfg["gf_method"]:
        orc.set_gf_groups([x.shape[0] for x in sf_all], [x.shape[0] for x in cs_all])
    try:
        return orc.scan2map(wl["surf_map"], wl["corner_map"], np.concatenate(sf_all), np.concatenate(cs_all), fr["init"], o)
    finally:
        orc.set_gf_groups(None, None)


def cpu_reference_arm(orc, cfg, wl, steps, warmup, time_cap_s=None):
    """The reference's CPU path on whole rig frames: per-LiDAR extractCloud under OpenMP (estimator.cpp:249), single-threaded
    mapper (kd-tree build every frame, matching, solve), kd-tree = the reference's own nanoflann when oracle/_ref is present.
    Returns (rig frames/s, threads used, per-frame seconds, last (pose, stats), kd-tree backend)."""
    L = cfg["lidars"]
    ncores = os.cpu_count() or 1
    threads = max(1, min(L, ncores))
    orc.set_threads(threads)
    ref_tree = orc.use_ref_tree(True)
    frames = wl["frames"]

    def run(fr):
        t = time.perf_counter()
        out = oracle_frame(orc, cfg, wl, fr, sharded=False)
        return time.perf_counter() - t, out

    try:
        for w in range(warmup):
            run(frames[w % len(frames)])
        times, last = [], None
        for k in range(steps):
            dt, last = run(frames[k % len(frames)])
            times.append(dt)
            if time_cap_s is not None and sum(times) > time_cap_s:  # bounded sample: stop early, report the steps done
                break
    finally:
        orc.use_ref_tree(False)
        orc.set_threads(1)
    return len(times) / sum(times), threads, times, last, ("reference nanoflann (oracle/_ref/libref_knn.so)" if ref_tree else "oracle restatement")


def gpu_measure(m, syn, torch, dist, cfg_name, cfg, args, rank, local_rank, world, steps, warmup, n_frames, full: bool):
    """Time one configuration on this process group.  Returns the per-rank measurement dict (rank 0 adds parity / baselines)."""
    n_gpus = world
    L = cfg["lidars"]
    p = m.default_params()
    p.n_scans, p.max_outer, p.max_inner, p.map_cell = cfg["rings"], cfg["gn_iters"], 1, args.map_cell
    p.max_ring_points = cfg["horizon"]
    p.gf_method, p.gf_ratio, p.gf_seed = cfg["gf_method"], cfg["gf_ratio"], 0
    ctx = m.Context(local_rank, p)
    exchange = None
    if world > 1:
        uid = [m.Context.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        ctx.comm_init(world, rank, uid[0])
        # peer-memory exchange inside the k_linearize tail when every GPU can map every other (NVLink / NVSwitch); the
        # NCCL all-reduce path stays as the fallback (MLOAM_DISABLE_P2P=1 forces it)
        can = all(torch.cuda.can_device_access_peer(local_rank, q) for q in range(world) if q != local_rank)
        flag = torch.tensor([1 if (can and os.environ.get("MLOAM_DISABLE_P2P", "0") in ("", "0")) else 0], device=torch.device("cuda", local_rank))
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if int(flag.item()) == 1:
            handles = [None] * world
            dist.all_gather_object(handles, ctx.comm_p2p_export())
            ctx.comm_p2p_init(world, rank, handles)
            exchange = "peer-memory stores + flags inside the k_linearize tail (NVLink), sum in rank order"
        else:
            exchange = "ncclAllReduce of the packed normal equations between the partial-sum and LM-step kernels"
        dist.barrier()
        torch.cuda.synchronize()

    wl = make_workload(syn, cfg, n_gpus, rank, n_frames, args.map)
    frames = wl["frames"]
    my = [f["groups"][rank] for f in frames]
    ids = wl["groups"][rank]
    if L > 1:
        ctx.set_lidars(len(ids), my[0]["ext"])
    n_scans = cfg["rings"] * len(ids)
    surf_map, corner_map = wl["surf_map"], wl["corner_map"]
    dev = torch.device("cuda", local_rank)
    d_surf = torch.from_numpy(surf_map).to(dev)
    d_corner = torch.from_numpy(corner_map).to(dev)
    d_frames = [dict(cloud=torch.from_numpy(g["cloud"]).to(dev), ss=torch.from_numpy(g["ss"]).to(dev), se=torch.from_numpy(g["se"]).to(dev)) for g in my]
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
    h_surf = torch.from_numpy(surf_map).pin_memory()
    h_corner = torch.from_numpy(corner_map).pin_memory()
    h_frames = [dict(cloud=torch.from_numpy(g["cloud"]).pin_memory(), ss=np.ascontiguousarray(g["ss"], np.int32), se=np.ascontiguousarray(g["se"], np.int32)) for g in my]
    for hf in h_frames:
        hf["cloud_np"] = hf["cloud"].numpy()  # one view per buffer: the look-ahead matches the announced sweep by its pointer
    h_surf_np, h_corner_np = h_surf.numpy(), h_corner.numpy()
    KF = max(1, args.keyframe_every)

    lookahead = not args.no_lookahead

    def step_device(k, rebuild):
        f, g, d = frames[k % n_frames], my[k % n_frames], d_frames[k % n_frames]
        if lookahead:  # announce sweep k+1: it is extracted on a side stream while frame k is matched and solved
            gn, dn = my[(k + 1) % n_frames], d_frames[(k + 1) % n_frames]
            ctx.frame_set_next_device(dn["cloud"].data_ptr(), gn["cloud"].shape[0], dn["ss"].data_ptr(), dn["se"].data_ptr(), n_scans)
        return ctx.frame_device(d["cloud"].data_ptr(), g["cloud"].shape[0], d["ss"].data_ptr(), d["se"].data_ptr(), n_scans,
                                d_surf.data_ptr(), surf_map.shape[0], d_corner.data_ptr(), corner_map.shape[0], f["init"], rebuild)

    def step_host(k, rebuild):
        f, hf = frames[k % n_frames], h_frames[k % n_frames]
        if lookahead:
            hn = h_frames[(k + 1) % n_frames]
            ctx.frame_set_next(hn["cloud_np"], hn["ss"], hn["se"])
        return ctx.frame(hf["cloud_np"], hf["ss"], hf["se"], h_surf_np, h_corner_np, f["init"], rebuild)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    stream = torch.cuda.Stream(device=dev)
    ctx.set_stream(stream.cuda_stream)
    sampler = ClockSampler(local_rank)
    sampler.start()
    sampler.wait_first()
    # warm-up: every (frame buffer, rebuild?) combination at least three times (first sighting allocates, the second captures
    # its CUDA graph, the third replays) so that no capture falls into the timed region; at least W steps in total
    # (with look-ahead the graph of a frame also depends on which half of the feature double buffer it uses, which alternates along an
    # unbroken k -> k+1 chain: n_frames is even, so the chain below visits every combination the timed loop will)
    n_warm = 0
    for rb in (True, False):
        for _ in range(4):
            for k in range(n_frames):
                step_device(k, rb)
                n_warm += 1
    for k in range(n_frames * ((max(0, warmup - n_warm) + n_frames - 1) // n_frames)):
        step_device(k, False)
    for k in range(n_frames):
        step_device(k, k == n_frames - 1)  # leave the resident maps freshly built; the chain continues into the timed loop at k = 0
    barrier()
    sampler.mark()
    launches0 = ctx.launch_count()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    last, feats, bad_term = None, 0, 0
    with torch.cuda.stream(stream):
        for k in range(steps):
            flush.fill_(k & 0xFF)  # not timed: evict the previous step's lines from L2
            if world > 1:
                dist.barrier()
            evs[k][0].record(stream)
            last = step_device(k, k % KF == 0)
            evs[k][1].record(stream)
            feats += last[1]["n_surf_in"] + last[1]["n_corner_in"]
            bad_term += 1 if last[1]["termination"] == 9 else 0
    barrier()
    clocks = sampler.stop()
    launches = ctx.launch_count() - launches0
    ms_steps = [a.elapsed_time(b) for a, b in evs]
    srt = sorted(ms_steps)
    res = dict(step_stats={"min": srt[0], "median": srt[len(srt) // 2], "p90": srt[int(0.9 * (len(srt) - 1))], "max": srt[-1]},
               keyframe_ms=statistics.mean(ms_steps[0::KF]), clocks=clocks, launches=int(launches), exchange=exchange, exchange_timeouts=bad_term,
               features_per_step=feats / steps, last_pose=last[0], last_stats=last[1], k_last=(steps - 1) % n_frames, wl=wl)
    if KF > 1 and steps > 1:
        rest = [x for i, x in enumerate(ms_steps) if i % KF]
        res["regular_ms"] = statistics.mean(rest) if rest else None
    t_max = sum(ms_steps) / 1e3
    if world > 1:
        tt = torch.tensor([t_max], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        t_max = float(tt.item())
    res["t_max"] = t_max
    res["value"] = L * steps / t_max

    # ---- per-kernel device times: the same schedule with the library's CUDA-event scopes (stream launches, not graph replay)
    if full:
        prof_steps = max(KF, min(steps, 20))
        ctx.profile(True)
        ctx.profile_reset()
        feats_prof, rebuilds = 0, 0
        with torch.cuda.stream(stream):
            for k in range(prof_steps):
                flush.fill_(k & 0xFF)
                st_k = step_device(k, k % KF == 0)[1]
                rebuilds += 1 if k % KF == 0 else 0
                feats_prof += st_k["n_surf_in"] + st_k["n_corner_in"]
        barrier()
        names = ("map_build", "extract", "voxel", "match", "fit", "linearize", "lm", "lm_tail_reduce", "lm_tail_advance")
        prof = {name: ctx.profile_get(name) for name in names}
        kp = {name: ctx.profile_get(name)[1] / prof_steps for name in ("knn_keep_matched", "knn_keep_rejected", "knn_ball", "knn_blind")}
        kp["max_query_cycles"] = ctx.profile_get("knn_max_query_cycles")[1]
        kp["queries_over_32k_cycles"] = ctx.profile_get("knn_queries_over_32k_cycles")[1] / prof_steps
        ctx.profile(False)
        res.update(prof=prof, prof_steps=prof_steps, prof_rebuilds=rebuilds, feats_prof=feats_prof, knn_paths=kp)
        # the map build alone (the streaming kernel of the path): its 8 launches captured into one CUDA graph — as inside the frame
        # graph — so that the events bracket device time, not host launch gaps; inputs resident, L2 flushed before every build
        for _ in range(3):
            ctx.map_build_device(1, d_surf.data_ptr(), surf_map.shape[0], args.map_cell)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=stream):
            ctx.map_build_device(1, d_surf.data_ptr(), surf_map.shape[0], args.map_cell)
        with torch.cuda.stream(stream):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            reps, t_b = 10, 0.0
            for r in range(reps):
                flush.fill_(r & 0xFF)
                e0.record(stream)
                graph.replay()
                e1.record(stream)
                torch.cuda.synchronize()
                t_b += e0.elapsed_time(e1)
        del graph
        res["map_build_ms"] = t_b / reps
        res["map_build_points"] = int(surf_map.shape[0])

    # ---- e2e: HOST buffers through the C ABI (H2D sweeps every step, both submaps on keyframe steps, D2H pose + state)
    e2e_steps = max(KF, steps) if full else max(KF, min(steps, 20))
    for rb in (True, False):
        for _ in range(4):
            for k in range(n_frames):
                step_host(k, rb)
    for k in range(n_frames):
        step_host(k, k == n_frames - 1)
    barrier()
    t0 = time.perf_counter()
    for k in range(e2e_steps):
        step_host(k, k % KF == 0)
    torch.cuda.synchronize()
    t_e2e = time.perf_counter() - t0
    if world > 1:
        tt = torch.tensor([t_e2e], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        t_e2e = float(tt.item())
    sweep_bytes = int(np.mean([g["cloud"].nbytes for g in my])) + 2 * n_scans * 4 + 7 * 8
    map_bytes = int(surf_map.nbytes + corner_map.nbytes)
    n_kf = len(range(0, e2e_steps, KF))
    res["e2e"] = {"value": L * e2e_steps / t_e2e, "unit": "frames/s", "h2d_bytes_per_step": int(sweep_bytes + map_bytes * n_kf / e2e_steps),
                  "d2h_bytes_per_step": int(7 * 8 + 4 * 2 + 1304), "steps": e2e_steps,
                  "h2d_detail": {"sweeps_every_step": sweep_bytes, "submaps_on_keyframe_steps": map_bytes, "keyframe_steps": n_kf}}
    ctx.close()
    return res


def dump_outputs(out_dir: str, R: dict, calib: bool) -> None:
    """--dump-outputs: what the timed call returned in its last timed step (the solved pose, or pose_i and ext_cal of a calibration
    step, and every field of the solve statistics), one float64 DIR/<name>.npy each.  The workload is seeded, so two builds run
    with the same arguments can be compared file by file."""
    outs = {"pose_i": R["last_pose"], "ext_cal": R["last_ext"]} if calib else {"pose": R["last_pose"]}
    outs.update((k, R["last_stats"][k]) for k in SOLVE_STATS)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in outs.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, np.float64))


def config_blurb(name, cfg, n_gpus, args, wl):
    per = max(1, cfg["lidars"] // n_gpus)
    return {"workload": f"{name}: {cfg['lidars']} LiDAR(s) x {cfg['rings']}-ring x {cfg['horizon']} sweep, {cfg['map_points']}-pt edge+surf submap (1:9), "
                        f"{cfg['gn_iters']} GN iterations (re-association each)" + (f", greedy good-feature selection {cfg['gf_ratio']}" if cfg["gf_method"] else "")
                        + (", 12-DoF online extrinsic calibration" if cfg["calib"] else ""),
            "lidars": cfg["lidars"], "rings": cfg["rings"], "horizon": cfg["horizon"], "map_points": cfg["map_points"], "gn_iters": cfg["gn_iters"],
            "gf_method": cfg["gf_method"], "gf_ratio": cfg["gf_ratio"], "parallelism": f"{per} LiDAR(s) per GPU x {n_gpus} GPU(s), submap replicated",
            "submap": wl["map_info"], "keyframe_every": args.keyframe_every,
            "schedule": f"submap uploaded + rebuilt on keyframe steps only (every {args.keyframe_every}th: DISTANCE_KEYFRAMES 1 m at 1 m/s, 10 Hz; "
                        "lidar_mapper_keyframe.cpp:1101), resident in HBM in between; the CPU arm rebuilds its kd-trees every frame as the reference does (:433-434)",
            "map_cell": args.map_cell if args.map_cell > 0 else "auto (per map, from the occupancy of the previous build)",
            "l2": "256 MiB buffer written between timed steps (L2 flush)"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default=None, choices=sorted(CONFIGS))
    ap.add_argument("--map", default="keyframes", choices=["keyframes", "uniform"])
    ap.add_argument("--map-cell", type=float, default=0.0, help="grid cell edge [m]; 0 = auto per map")
    ap.add_argument("--keyframe-every", type=int, default=KEYFRAME_EVERY)
    ap.add_argument("--cpu-sample", type=int, default=0, help="rig frames of CPU work for cpu_baseline (0: ~10-30 s worth)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-lookahead", action="store_true", help="do not announce sweep k+1 while frame k runs (no overlap of extraction with the solve)")
    ap.add_argument("--no-c4", action="store_true", help="skip the extra C4-on-one-GPU measurement of the default run")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step returned as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs records the GPU arm (--impl ours)")

    if args.gpus > 1 and "WORLD_SIZE" not in os.environ and args.impl == "ours":
        # N > 1 is one process per GPU: when not already under torchrun, relaunch this command under it
        import socket

        with socket.socket() as sk:
            sk.bind(("127.0.0.1", 0))
            port = sk.getsockname()[1]
        os.execv(sys.executable, [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(args.gpus),
                                  "--master-addr", "127.0.0.1", "--master-port", str(port), os.path.abspath(__file__)] + sys.argv[1:])
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    n_gpus = args.gpus
    import synthetic as syn

    cfg_name = args.config or DEFAULT_CONFIG.get(n_gpus, "C2")
    cfg = dict(CONFIGS[cfg_name])
    if cfg["lidars"] % n_gpus != 0:  # e.g. C2 forced onto several GPUs: one such LiDAR per GPU ("C2-like x N")
        cfg["lidars"] = n_gpus
    L = cfg["lidars"]

    # ------------------------------------------------------------------ reference arm (CPU)
    if args.impl == "reference":
        if rank != 0:
            return 0
        import oracle_lib as orc
        n_frames = max(1, min(args.steps, 3))
        warm = max(0, min(args.warmup, 1))
        if cfg["calib"]:
            from bench_calib import cpu_calib_arm, make_calib_workload
            cases, map_info = make_calib_workload(syn, cfg, n_frames, args.map)
            wl = {"map_info": map_info}
            fps_rig, times, _, tree = cpu_calib_arm(orc, cfg, cases, max(1, args.steps), time_cap_s=150.0)
            threads = 1
        else:
            wl = make_workload(syn, cfg, 1, 0, n_frames, args.map)
            fps_rig, threads, times, _, tree = cpu_reference_arm(orc, cfg, wl, max(1, args.steps), warm, time_cap_s=150.0)
        steps = len(times)
        value = L * fps_rig
        sample = (f"{steps} rig frame(s) of {cfg_name} ({L} LiDAR sweep(s) each, {sum(times):.1f} s of CPU work): CPU restatement of the reference path "
                  f"(oracle/, -O3 -march=x86-64-v3), kd-tree build + search = {tree}; threading as the reference: extractCloud under OpenMP over the "
                  f"LiDARs ({threads} thread(s)), mapper single-threaded, kd-trees rebuilt every frame; host has {os.cpu_count()} logical cores")
        line = {"metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": n_gpus, "steps": steps, "warmup": warm,
                "ms_per_step": 1e3 * sum(times) / len(times), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32/f64", "data": "synthetic", "impl": "reference", "config": config_blurb(cfg_name, cfg, n_gpus, args, wl),
                "cpu_baseline": {"value": value, "unit": "frames/s", "cores": threads, "kind": "port", "sample": sample},
                "e2e": {"value": value, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return 0

    # ------------------------------------------------------------------ our arm (GPU)
    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        print(json.dumps({"error": "no CUDA device: this framework has no CPU path"}))
        return 2
    torch.cuda.set_device(local_rank)
    saved_stdout = None
    if world > 1:
        # NCCL may print its version banner on stdout: the contract is ONE JSON line, so C-level stdout points at stderr meanwhile
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    m = load_mloam()
    n_frames = 8 if L == 1 else 4
    try:
        if cfg["calib"]:
            from bench_calib import gpu_measure_calib
            R = gpu_measure_calib(m, syn, torch, dist, cfg_name, cfg, args, rank, local_rank, world, args.steps, args.warmup, n_frames)
        else:
            R = gpu_measure(m, syn, torch, dist, cfg_name, cfg, args, rank, local_rank, world, args.steps, args.warmup, n_frames, full=True)
    finally:
        if saved_stdout is not None:
            sys.stdout.flush()
            os.dup2(saved_stdout, 1)
            os.close(saved_stdout)
    # ---- N > 1: the BASELINE configurations differ from N to N (calibration at 2, 128 rings + feature selection at 8), so their
    # values do not form a scaling curve.  A compact second measurement keeps one: the same number of 64-ring LiDARs as GPUs,
    # plain scan2MapOptimization, the configuration's submap size ("C2-like x N", what round 1 reported).
    probe = None
    if world > 1 and (cfg["calib"] or cfg["gf_method"] or cfg["rings"] != 64):
        pc = dict(CONFIGS["C2"], lidars=world, map_points=cfg["map_points"])
        saved = None
        if rank == 0:
            sys.stdout.flush()
            saved = os.dup(1)
            os.dup2(2, 1)
        try:
            P = gpu_measure(m, syn, torch, dist, "C2-like", pc, args, rank, local_rank, world, min(args.steps, 20), args.warmup, 4, full=False)
        finally:
            if saved is not None:
                sys.stdout.flush()
                os.dup2(saved, 1)
                os.close(saved)
        probe = {"workload": f"C2-like x {world}: one 64-ring x 2048 LiDAR per GPU, {pc['map_points']}-pt submap, 10 GN iterations, no calibration / feature selection",
                 "value": P["value"], "unit": "frames/s", "ms_per_step": 1e3 * P["t_max"] / min(args.steps, 20), "e2e": P["e2e"], "exchange": P["exchange"],
                 "exchange_timeouts": P["exchange_timeouts"]}
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, R, cfg["calib"])

    wl = R["wl"]
    config = config_blurb(cfg_name, cfg, n_gpus, args, wl)
    if R.get("exchange"):
        config["exchange"] = R["exchange"]
    if not cfg["calib"]:
        config["lookahead"] = ("off" if args.no_lookahead else
                           "sweep k+1 is announced with frame k (mloam_frame_set_next*): its extractCloud + scan down-sampling run on a side stream while frame k "
                           "is matched and solved, and are joined before frame k returns — every timed step contains one extraction and one solve "
                           "(the reference overlaps the same stages across its estimator and lidar_mapper nodes)")
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (burst copy)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    roofline, stage_ms = None, None
    if "prof" in R:
        prof, ps = R["prof"], R["prof_steps"]
        match_ms, match_launches = prof["match"]
        alg = R["feats_prof"] * cfg["gn_iters"] * KNN_BYTES_PER_FEATURE
        ach = (alg / 1e9) / (match_ms / 1e3) if match_ms > 0 else 0.0
        traffic = None
        tp = os.path.join(ROOT, "profiles", "r02_match_traffic.json")
        if os.path.exists(tp):
            try:
                traffic = json.load(open(tp)).get("dram_bytes_per_launch")
            except Exception:
                traffic = None
        roofline = {"bound": "hbm", "kernel": "k_match_knn<5> (pointAssociateToMap + exact 5-NN over the dense voxel grid, one warp per feature, TMA-staged rows)",
                    "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": traffic, "peak_source": peak_src,
                    "algorithmic_bytes_per_feature": KNN_BYTES_PER_FEATURE, "avg_launch_us": 1e3 * match_ms / max(1, match_launches), "launches": match_launches,
                    "note": "the submap is L2-resident and a launch moves ~1 MB of compulsory bytes: latency-bound, not HBM-bound (DESIGN.md 4)"}
        mb_ach = R["map_build_points"] * MAP_BYTES_PER_POINT / 1e9 / (R["map_build_ms"] / 1e3)
        roofline_map = {"bound": "hbm", "kernel": "map build (k_grid_bbox + k_grid_count + k_grid_scan_a/b + k_grid_scatter: counting sort into the dense grid)",
                        "achieved": mb_ach, "peak": peak, "unit": "GB/s", "frac": mb_ach / peak, "traffic": None, "peak_source": peak_src,
                        "algorithmic_bytes_per_point": MAP_BYTES_PER_POINT, "points": R["map_build_points"], "avg_build_us": 1e3 * R["map_build_ms"]}
        stage_ms = {k: v[0] / ps for k, v in prof.items()}
    # ---- pose parity of the last timed frame against the oracle, at every N (sharded restatement for N > 1)
    import oracle_lib as orc
    parity = None
    if not cfg["calib"]:
        k_last = R["k_last"]
        fr = wl["frames"][k_last]
        if world > 1:  # the other ranks' sweeps of that frame
            wl_all = make_workload(syn, cfg, n_gpus, 0, n_frames, args.map, all_groups=True)
            fr = wl_all["frames"][k_last]
        ref_pose, ref_st = oracle_frame(orc, cfg, wl, fr, sharded=world > 1)
        dt, dr = syn.pose_err(R["last_pose"], ref_pose)
        parity = {"m": dt, "rad": dr, "matches_gpu": [R["last_stats"]["n_surf"], R["last_stats"]["n_corner"]],
                  "matches_oracle": [int(ref_st["n_surf"]), int(ref_st["n_corner"])], "frame": int(k_last)}
        config["pose_err_vs_oracle"] = parity
    else:
        config["pose_err_vs_oracle"] = R.get("parity")
    # ---- cpu_baseline (N = 1 only): bounded sample of the same workload
    cpu = None
    if not args.no_cpu_baseline and world == 1 and cfg["calib"]:
        from bench_calib import cpu_calib_arm
        fps_rig, times, _, tree = cpu_calib_arm(orc, cfg, wl["cases"], 6, time_cap_s=30.0)
        cpu = {"value": L * fps_rig, "unit": "frames/s", "cores": 1, "kind": "port",
               "sample": f"{len(times)} calibration step(s) of this workload ({sum(times):.1f} s of CPU work), CPU restatement (-O3), kd-tree = {tree}, single-threaded as the reference"}
    elif not args.no_cpu_baseline and world == 1:
        est = 0.6 * L * cfg["map_points"] / 1e6 + 0.3  # ~s per rig frame on one core
        n_cpu = args.cpu_sample or max(2, min(12, int(round(15.0 / est))))
        fps_rig, threads, times, _, tree = cpu_reference_arm(orc, cfg, wl, n_cpu, 1, time_cap_s=40.0)
        cpu = {"value": L * fps_rig, "unit": "frames/s", "cores": threads, "kind": "port",
               "sample": f"{len(times)} rig frame(s) of this workload ({sum(times):.1f} s of CPU work), CPU restatement of the reference path (-O3), kd-tree = {tree}, "
                         f"reference threading (extractCloud under OpenMP over the LiDARs, single-threaded mapper, kd-trees rebuilt every frame); host has {os.cpu_count()} logical cores"}

    line = {"metric": METRIC, "value": R["value"], "unit": "frames/s", "n_gpus": n_gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * R["t_max"] / args.steps, "ms_per_step_stats": R["step_stats"], "ms_keyframe_step": R.get("keyframe_ms"), "ms_regular_step": R.get("regular_ms"),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32/f64", "data": "synthetic", "config": config,
            "ms_per_gn_iter": 1e3 * R["t_max"] / args.steps / cfg["gn_iters"], "e2e": R["e2e"], "gpu_launches": R["launches"],
            "cuda_graph_replay": os.environ.get("MLOAM_DISABLE_GRAPHS", "0") in ("", "0") and (world == 1 or "peer-memory" in (R.get("exchange") or "")),
            "clocks": R["clocks"], "features_per_step": R["features_per_step"], "exchange_timeouts": R["exchange_timeouts"]}
    if roofline:
        line["roofline"] = roofline
        line["roofline_map_build"] = roofline_map
        line["stage_ms_per_step"] = stage_ms
        line["knn_queries_per_step_by_path"] = R["knn_paths"]
    if cpu is not None:
        line["cpu_baseline"] = cpu
    if probe is not None:
        line["weak_scaling_probe"] = probe
    # ---- the north star's target configuration next to the default one: C4 (4 x 64-ring LiDARs, 5M-point submap) on ONE GPU
    if world == 1 and cfg_name == "C2" and not args.no_c4:
        c4 = dict(CONFIGS["C4"])
        R4 = gpu_measure(m, syn, torch, dist, "C4", c4, args, 0, local_rank, 1, min(args.steps, 20), args.warmup, 4, full=False)
        fr4 = R4["wl"]["frames"][R4["k_last"]]
        ref4, st4 = oracle_frame(orc, c4, R4["wl"], fr4, sharded=False)
        dt4, dr4 = syn.pose_err(R4["last_pose"], ref4)
        entry = {"workload": config_blurb("C4", c4, 1, args, R4["wl"])["workload"] + " — all four LiDARs batched in one context on ONE GPU",
                 "value": R4["value"], "unit": "frames/s (LiDAR sweeps; rig frames/s = value / 4)", "ms_per_rig_frame": 1e3 * R4["t_max"] / min(args.steps, 20),
                 "ms_per_step_stats": R4["step_stats"], "e2e": R4["e2e"], "pose_err_vs_oracle": {"m": dt4, "rad": dr4}, "gpu_launches": R4["launches"],
                 "features_per_step": R4["features_per_step"]}
        if not args.no_cpu_baseline:
            fps_rig, threads, times, _, tree = cpu_reference_arm(orc, c4, R4["wl"], 3, 0, time_cap_s=30.0)
            entry["cpu_baseline"] = {"value": 4 * fps_rig, "unit": "frames/s", "cores": threads, "kind": "port",
                                     "sample": f"{len(times)} rig frame(s) ({sum(times):.1f} s of CPU work), kd-tree = {tree}, reference threading"}
            entry["e2e_vs_cpu"] = R4["e2e"]["value"] / (4 * fps_rig)
        line["c4_one_gpu"] = entry
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 3 if R["exchange_timeouts"] else 0


if __name__ == "__main__":
    sys.exit(main())
