"""N>1 path on real GPUs (needs >= 2 visible devices, otherwise skipped): two NCCL ranks shard the frame windows of one
video (dist_mode="windows": cached CUDA-graph session per rank, ReferenceNet banks broadcast from rank 0 as ONE flat buffer,
one fp32 sum all-reduce of the accumulated noise prediction per step, decoded frames all-gathered) and must reproduce the
single-process result; dist_mode="clips" (the
weak-scaling mode bench.py uses for N>1) must leave every rank with its own, locally computed video."""
import os
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "golden")


def _worker(rank, world, port, q):
    sys.path.insert(0, HERE)
    sys.path.insert(0, os.path.dirname(HERE))
    import torch.distributed as dist
    from helpers import build_pipeline, pipeline_inputs
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    gold = torch.load(os.path.join(GOLDEN, "pipeline_small.pt"))
    P = gold["params"]
    L = 24                                                  # two overlapping 16-frame windows -> one per rank
    pipe = build_pipeline(P, dev)
    ref_image, poses, ref_pose = pipeline_inputs(P["size"], L, P["seeds"]["inputs"])
    g = torch.manual_seed(5)
    lat0 = torch.randn((1, 4, L, P["size"] // 8, P["size"] // 8), generator=g).to(torch.float16)
    args = (ref_image, poses, ref_pose, P["size"], P["size"], L, 3, P["guidance"])
    single = pipe(*args, latents=lat0.clone()).videos if rank == 0 else None
    single_lat = pipe.last_latents.float().cpu() if rank == 0 else None
    sharded = pipe(*args, latents=lat0.clone(), dist_mode="windows").videos      # builds + captures the sharded session
    sharded_lat = pipe.last_latents.float().cpu()
    again = pipe(*args, latents=lat0.clone(), dist_mode="windows").videos        # pure replay: rank-0 write graph, ONE flat
    assert torch.equal(again, sharded)                                           # bank broadcast, read graph, unit graphs
    assert torch.equal(pipe.last_latents.float().cpu(), sharded_lat)
    pipe.collect_timings()
    assert pipe.timings.get("bank_broadcast_ms", 0.0) > 0.0 and pipe.timings.get("all_reduce_ms", 0.0) > 0.0
    pipe(*args, latents=lat0.clone(), dist_mode="window_branches")        # (window, CFG branch) units: 4 units on 2 ranks,
    branch_lat = pipe.last_latents.float().cpu()                          # batched into one UNet call per rank (group_units)
    pipe.group_units = 0                                                   # the same with one call per unit
    pipe(*args, latents=lat0.clone(), dist_mode="window_branches")
    ungrouped_lat = pipe.last_latents.float().cpu()
    pipe.group_units = 4
    assert float((ungrouped_lat - branch_lat).norm() / branch_lat.norm()) < 5e-3
    # clips mode: every rank runs its own clip end to end (rank-dependent noise), no data-path collective
    lat_r = torch.randn((1, 4, L, P["size"] // 8, P["size"] // 8), generator=torch.manual_seed(100 + rank)).to(torch.float16)
    clips = pipe(*args, latents=lat_r.clone(), dist_mode="clips").videos
    own = pipe(*args, latents=lat_r.clone()).videos
    torch.cuda.synchronize()
    q.put((rank, single, single_lat, sharded, sharded_lat, float((clips - own).norm() / own.norm()), branch_lat))
    dist.barrier()
    dist.destroy_process_group()


def test_window_sharding_two_gpus_nccl():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    from helpers import rel_l2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, 2, 29541, q)) for r in range(2)]
    for p in procs:
        p.start()
    got = {}
    for _ in range(2):
        r = q.get(timeout=600)
        got[r[0]] = r
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    _, single, single_lat, sh0, sh0_lat, clip_err0, br0_lat = got[0]
    _, _, _, sh1, sh1_lat, clip_err1, br1_lat = got[1]
    # both ranks hold the same latents / video after the all-reduce + all-gather
    assert torch.equal(sh0_lat, sh1_lat)
    assert torch.equal(sh0, sh1)
    e_lat = rel_l2(sh0_lat, single_lat)
    e_vid = rel_l2(sh0, single)
    print(f"2-GPU window sharding vs single process: latents {e_lat:.3e}, video {e_vid:.3e}")
    # same kernels, same per-window results; each accumulator element receives at most one contribution per rank, so the
    # NCCL sum is exact as well
    assert e_lat < 1e-6 and e_vid < 1e-6
    assert clip_err0 < 1e-6 and clip_err1 < 1e-6
    # branch units run batch-1 UNet calls: same math, but GroupNorm's partial-sum chunking depends on the frame count of
    # the call, so the result matches the single-process one to rounding, not bit for bit
    assert torch.equal(br0_lat, br1_lat)
    e_br = rel_l2(br0_lat, single_lat)
    print(f"2-GPU (window, branch) units vs single process: latents {e_br:.3e}")
    assert e_br < 5e-3
