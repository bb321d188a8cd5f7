"""N > 1 coverage.  CPU (gloo, world_size 2): the property the GPU path relies on — the per-LiDAR normal equations
summed by an all-reduce equal the normal equations of the merged features — and the bench's rank-invariant workload.
GPU: tests/multi_gpu_check.py under torch.distributed.run when >= 2 GPUs are visible."""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _gloo_worker(rank, world, port, ret):
    import torch
    import torch.distributed as dist

    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as orc
    import synthetic as syn

    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    scene = syn.make_scene()
    truth = syn.trajectory(3)[2]
    surf_map, corner_map = syn.make_submap(scene, 30000)
    init = syn.perturb_pose(truth, np.random.Generator(np.random.PCG64(5)))
    feats = []
    for r in range(world):
        cloud, ss, se = syn.make_sweep(scene, truth, 16, 512, seed=60, lidar_id=r)
        f = orc.extract_cloud(cloud, ss, se)
        feats.append(orc.voxel_grid(f["surf_points_less_flat"], 0.4, True)[0])

    def ne(sf):
        v, cf, _ = orc.match_from_map("s", surf_map, sf, init)
        types = np.full(int(v.sum()), ord("s"), np.uint8)
        return orc.normal_eq(types, sf[v][:, :3].astype(np.float64), cf[v], 1.0, 0.1, init)

    H, g, cost = ne(feats[rank])  # this rank's LiDAR
    packed = torch.from_numpy(np.concatenate([H.reshape(-1), g, [cost]]))
    dist.all_reduce(packed)  # the single collective of the path
    Hm, gm, costm = ne(np.concatenate(feats))  # merged features on one process
    merged = np.concatenate([Hm.reshape(-1), gm, [costm]])
    ok = np.allclose(packed.numpy(), merged, rtol=1e-12, atol=1e-9)
    ret[rank] = bool(ok)
    dist.destroy_process_group()


def test_allreduce_of_per_lidar_normal_equations_equals_merged_gloo():
    import torch.multiprocessing as mp

    world = 2
    with mp.Manager() as mgr:
        ret = mgr.dict()
        mp.spawn(_gloo_worker, args=(world, 29511, ret), nprocs=world, join=True)
        assert all(ret[r] for r in range(world))


def test_bench_workload_is_rank_invariant_where_it_must_be():
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import bench
    import synthetic as syn

    assert bench.lidar_extrinsic(syn, 0, 4) is None
    e1, e2 = bench.lidar_extrinsic(syn, 1, 4), bench.lidar_extrinsic(syn, 2, 4)
    assert abs(np.linalg.norm(e1[3:]) - 1) < 1e-12 and not np.allclose(e1, e2)
    cfg = dict(bench.CONFIGS["C4"], rings=16, horizon=256, map_points=20000)  # small for the test
    w0 = bench.make_workload(syn, cfg, 2, 0, 2, "uniform")
    w1 = bench.make_workload(syn, cfg, 2, 1, 2, "uniform")
    assert np.array_equal(w0["surf_map"], w1["surf_map"]) and np.array_equal(w0["corner_map"], w1["corner_map"])  # replicated submap
    assert all(np.array_equal(a["init"], b["init"]) for a, b in zip(w0["frames"], w1["frames"]))  # shared LM state starts identical
    assert w0["groups"] == [[0, 1], [2, 3]]                                                    # LiDARs sharded in consecutive groups
    g0, g1 = w0["frames"][0]["groups"][0], w1["frames"][0]["groups"][1]
    assert not np.array_equal(g0["cloud"][:100], g1["cloud"][:100]) and g0["ext"].shape == (2, 7) and g0["ss"].shape[0] == 32
    # rank 0 can rebuild every group's sweeps for the per-N parity check; they equal what the other rank generated
    wa = bench.make_workload(syn, cfg, 2, 0, 2, "uniform", all_groups=True)
    assert np.array_equal(wa["frames"][0]["groups"][1]["cloud"], g1["cloud"])


@pytest.mark.gpu
@pytest.mark.parametrize("exchange", ["p2p", "nccl"])
def test_two_gpu_frame_parity(exchange):
    """Both exchanges of the packed normal equations: peer-memory stores inside the k_linearize tail, NCCL all-reduce."""
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs (runs tests/multi_gpu_check.py under torchrun on two of them)")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29533" if exchange == "p2p" else "29534", os.path.join(ROOT, "tests", "multi_gpu_check.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=dict(os.environ, MLOAM_EXCHANGE=exchange))
    assert out.returncode == 0 and "MULTI_GPU_CHECK OK" in out.stdout, out.stdout[-2000:] + out.stderr[-2000:]


@pytest.mark.gpu
def test_two_gpu_calibration_parity():
    """12-DoF online calibration sharded over two GPUs (one LiDAR each) with the NCCL all-reduce of the 12x12 normal equations."""
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs (runs tests/multi_gpu_calib_check.py under torchrun on two of them)")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29541", os.path.join(ROOT, "tests", "multi_gpu_calib_check.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "MULTI_GPU_CALIB_CHECK OK" in out.stdout, out.stdout[-2000:] + out.stderr[-2000:]


def test_peer_exchange_protocol_model():
    """Model of lm_tail's peer-memory exchange (solve_kernels.cu): per rank an exchange buffer with slots[2][N] and
    flags[2][N], double-buffered by epoch parity; a rank publishes its contribution into every rank's slot[parity][me],
    raises flag[parity][me] = epoch + 1 there, waits for all flags of its own buffer, sums the slots in rank order and
    only then moves on.  Run by N threads with random stalls: every rank must compute the identical (bit-identical) sum at
    every epoch and no slot may be overwritten before every reader has consumed it (ranks drift by at most one epoch)."""
    import random
    import threading
    import time

    for n_ranks in (2, 4, 8):
        epochs = 60
        rng = np.random.default_rng(7)
        contrib = rng.normal(size=(epochs, n_ranks, 30))  # what rank r contributes at epoch e
        slots = np.zeros((n_ranks, 2, n_ranks, 30))       # slots[owner][parity][from]
        flags = np.zeros((n_ranks, 2, n_ranks), np.int64)
        sums = np.zeros((n_ranks, epochs, 30))
        max_lead = [0]
        progress = [0] * n_ranks
        errors = []

        def rank_main(me):
            rnd = random.Random(100 + me)
            for e in range(epochs):
                par, target = e & 1, e + 1
                if rnd.random() < 0.3:
                    time.sleep(rnd.random() * 2e-3)
                for q in range(n_ranks):          # peer stores
                    slots[q, par, me] = contrib[e, me]
                for q in range(n_ranks):          # then the flags (the kernel fences in between)
                    flags[q, par, me] = target
                t0 = time.time()
                while not all(flags[me, par, q] >= target for q in range(n_ranks)):
                    if time.time() - t0 > 20:
                        errors.append(f"rank {me} timed out at epoch {e}")
                        return
                    time.sleep(0)
                acc = np.zeros(30)
                for q in range(n_ranks):          # rank order: identical on every rank
                    acc = acc + slots[me, par, q]
                sums[me, e] = acc
                progress[me] = e + 1
                max_lead[0] = max(max_lead[0], max(progress) - min(progress))

        threads = [threading.Thread(target=rank_main, args=(r,)) for r in range(n_ranks)]
        [t.start() for t in threads]
        [t.join() for t in threads]
        assert not errors, errors
        expect = np.zeros((epochs, 30))
        for e in range(epochs):
            acc = np.zeros(30)
            for q in range(n_ranks):
                acc = acc + contrib[e, q]
            expect[e] = acc
        for r in range(n_ranks):
            assert np.array_equal(sums[r], expect), f"rank {r} summed stale or torn slots"
        assert max_lead[0] <= 2  # published (epoch e+1) while the slowest still reads epoch e at most
