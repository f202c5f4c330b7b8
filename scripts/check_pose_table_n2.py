"""Two-GPU check of GraphedTrainStep(poses=...): each rank takes half of a seeded batch for 5 graphed steps; the pose
gradient is summed over the ranks in the step, so `se3` must end bitwise equal on both ranks and, within fp32 summation
order, equal to a one-GPU run on the whole batch.

The tolerance is measured, not assumed: rank 0 also runs the split on one GPU, eagerly (both halves' gradients accumulated
into .grad with the data-parallel loss scale, then both FusedAdam steps), which differs from the whole-batch run by summation
order only; the two-rank `se3` must lie within 4x that difference of the whole-batch run.  The pose bucket's allreduce is
timed on its own (CUDA events, median of 50).  Without torchrun (one process) the script runs the one-GPU part only and
reports the summation-order difference.

usage: torchrun --nproc_per_node 2 scripts/check_pose_table_n2.py [--out FILE]
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402


def run(rank, world, pxs, tgts, dev):
    from mvip_nerf_b200.cameras import CameraPoses
    from mvip_nerf_b200.graph import GraphedTrainStep
    from mvip_nerf_b200.optim import FusedAdam
    from mvip_nerf_b200.run import _FusedQuery
    from mvip_nerf_b200.run_nerf_helpers import NeRF, get_embedder
    torch.manual_seed(5)
    nc, nf = [NeRF(input_ch=63, input_ch_views=27, use_viewdirs=True).to(dev) for _ in range(2)]
    e, _ = get_embedder(10)
    ev, _ = get_embedder(4)
    kw = dict(network_query_fn=_FusedQuery(e, ev, 65536), network_fn=nc, network_fine=nf, N_samples=64, N_importance=64,
              perturb=0., raw_noise_std=0., white_bkgd=True, lindisp=True, use_viewdirs=True, ndc=False)
    g = torch.Generator().manual_seed(2)
    init = (torch.tensor([[1., 0, 0, 0.1], [0, 1, 0, -0.2], [0, 0, 1, 4.0]]) + 0.02 * torch.randn(6, 3, 4, generator=g)).to(dev)
    cam = CameraPoses(init)
    n = pxs[0].shape[0] // world
    step = GraphedTrainStep(kw, FusedAdam([p for m in (nc, nf) for p in m.parameters()], lr=5e-4), 64, 80, 70.0, n, 2.0, 6.0,
                            poses=cam, pose_optimizer=FusedAdam(cam.parameters(), lr=1e-3))
    for px, tgt in zip(pxs, tgts):
        step(px[rank * n:(rank + 1) * n], tgt[rank * n:(rank + 1) * n])
    torch.cuda.synchronize()
    return cam.se3.detach().clone()


def run_split(pxs, tgts, dev, world=2):
    """the data-parallel step on one GPU, eagerly: the gradients of `world` slices accumulated, then both Adam steps"""
    from mvip_nerf_b200 import run as mrun
    from mvip_nerf_b200.cameras import CameraPoses
    from mvip_nerf_b200.graph import default_loss
    from mvip_nerf_b200.optim import FusedAdam
    from mvip_nerf_b200.run import _FusedQuery
    from mvip_nerf_b200.run_nerf_helpers import NeRF, get_embedder
    torch.manual_seed(5)
    nc, nf = [NeRF(input_ch=63, input_ch_views=27, use_viewdirs=True).to(dev) for _ in range(2)]
    e, _ = get_embedder(10)
    ev, _ = get_embedder(4)
    kw = dict(network_query_fn=_FusedQuery(e, ev, 65536), network_fn=nc, network_fine=nf, N_samples=64, N_importance=64,
              perturb=0., raw_noise_std=0., white_bkgd=True, lindisp=True, use_viewdirs=True, ndc=False)
    g = torch.Generator().manual_seed(2)
    init = (torch.tensor([[1., 0, 0, 0.1], [0, 1, 0, -0.2], [0, 0, 1, 4.0]]) + 0.02 * torch.randn(6, 3, 4, generator=g)).to(dev)
    cam = CameraPoses(init)
    opt = FusedAdam([p for m in (nc, nf) for p in m.parameters()], lr=5e-4)
    popt = FusedAdam(cam.parameters(), lr=1e-3)
    n = pxs[0].shape[0] // world
    for px, tgt in zip(pxs, tgts):
        opt.zero_grad(set_to_none=True)
        popt.zero_grad(set_to_none=True)
        for r in range(world):
            t = tgt[r * n:(r + 1) * n]
            out = mrun.render(64, 80, 70.0, chunk=1024 * 32, c2w=cam(), pixels=px[r * n:(r + 1) * n], near=2.0, far=6.0,
                              _mse=(t, None), **kw)
            default_loss(*out, t, 1.0 / world).backward()
        opt.step()
        popt.step()
    torch.cuda.synchronize()
    return cam.se3.detach().clone()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    from mvip_nerf_b200 import dist as md
    rank, world, local = md.init_from_env()
    dev = torch.device("cuda", local)
    g = torch.Generator().manual_seed(3)
    N = 4096
    pxs = [torch.stack([torch.randint(6, (N,), generator=g), torch.randint(64, (N,), generator=g), torch.randint(80, (N,), generator=g)],
                       1).to(torch.int32).to(dev) for _ in range(5)]
    tgts = [torch.rand(N, 3, generator=g).to(dev) for _ in range(5)]
    res = {"world": world}
    if world > 1:
        se3 = run(rank, world, pxs, tgts, dev)
        both = [torch.empty_like(se3) for _ in range(world)]
        dist.all_gather(both, se3)
        res["se3_equal_on_ranks"] = all(torch.equal(both[0], b) for b in both)
        bucket = torch.randn(se3.numel(), device=dev)      # the pose bucket: V x 6 fp32
        for _ in range(5):
            dist.all_reduce(bucket)
        ts = []
        for _ in range(50):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            dist.all_reduce(bucket)
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        res["pose_bucket_allreduce_ms_median"] = sorted(ts)[len(ts) // 2]
        dist.destroy_process_group()     # the one-GPU runs below see world() == 1
        if rank != 0:
            return
    one = run(0, 1, pxs, tgts, dev)
    split = run_split(pxs, tgts, dev)
    order = float((one - split).abs().max())
    tol = 4 * max(order, 1e-7 * float(one.abs().max()))
    res.update({"se3_max_abs": float(one.abs().max()), "split_vs_whole_one_gpu": order, "tolerance": tol})
    ok = True
    if world > 1:
        diff = float((one - se3).abs().max())
        res.update({"two_gpu_vs_whole": diff, "two_gpu_vs_split": float((split - se3).abs().max())})
        ok = res["se3_equal_on_ranks"] and diff <= tol
    res["ok"] = ok
    print(json.dumps(res))
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
    sys.exit(0 if ok else 1)

if __name__ == "__main__":
    main()
