"""Times the pose-table training step on one GPU and merges the result into a JSON document (card name and power limit read in
the same run).

  * cfg 2 (4,096 rays, 64 + 64 samples, train kwargs) as a GraphedTrainStep, without poses (rays copied in) and with a 20-view
    CameraPoses table (pixels copied in), the two steps alternating in one process; per-step CUDA events, median and spread;
  * the pose module alone (forward + backward of CameraPoses, the small torch ops the graphed step runs for it), eager, and
    with the pose FusedAdam as a CUDA graph of its own (its share of the graphed step);
  * per-call times of the new entries (ops.kernel_timer, eager, same shapes).

usage: python scripts/time_pose_table.py [--out FILE] [--steps N] [--warmup W]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else torch.cuda.get_device_name()


def kwargs(nc, nf):
    from mvip_nerf_b200.run import _FusedQuery
    from mvip_nerf_b200.run_nerf_helpers import get_embedder
    e, _ = get_embedder(10)
    ev, _ = get_embedder(4)
    return dict(network_query_fn=_FusedQuery(e, ev, 65536), network_fn=nc, network_fine=nf, N_samples=64, N_importance=64,
                perturb=1., raw_noise_std=1., white_bkgd=False, lindisp=False, use_viewdirs=True, ndc=False)


def event_ms(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def stats(ts):
    ts = sorted(ts)
    return {"median_ms": ts[len(ts) // 2], "min_ms": ts[0], "max_ms": ts[-1], "n": len(ts)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    a = ap.parse_args()
    from mvip_nerf_b200 import ops
    from mvip_nerf_b200.cameras import CameraPoses
    from mvip_nerf_b200.graph import GraphedTrainStep
    from mvip_nerf_b200.optim import FusedAdam
    from mvip_nerf_b200.run_nerf_helpers import NeRF
    dev = torch.device("cuda", 0)
    H, W, focal, near, far, N, V = 756, 1008, 767.2935, 1.2, 7.7369, 4096, 20

    def nets(seed):
        torch.manual_seed(seed)
        return [NeRF(input_ch=63, input_ch_views=27, use_viewdirs=True).to(dev) for _ in range(2)]
    g = torch.Generator(device=dev).manual_seed(0)
    c0 = torch.tensor([[1., 0, 0, 0], [0, 1, 0, 0], [0, 0, 1, 4.0]], device=dev)
    init = c0.expand(V, 3, 4) + 0.01 * torch.randn(V, 3, 4, device=dev, generator=g)

    na = nets(1)
    step_rays = GraphedTrainStep(kwargs(*na), FusedAdam([p for n in na for p in n.parameters()], lr=5e-4), H, W, focal, N, near, far)
    nb = nets(1)
    cam = CameraPoses(init)
    step_pose = GraphedTrainStep(kwargs(*nb), FusedAdam([p for n in nb for p in n.parameters()], lr=5e-4), H, W, focal, N, near, far,
                                 poses=cam, pose_optimizer=FusedAdam(cam.parameters(), lr=1e-3))
    px = torch.stack([torch.randint(V, (N,), device=dev, generator=g), torch.randint(H, (N,), device=dev, generator=g),
                      torch.randint(W, (N,), device=dev, generator=g)], 1).to(torch.int32)
    rays_flat = ops.rays_from_poses(H, W, focal, init, px, near, far)
    rays = torch.stack([rays_flat[:, 0:3], rays_flat[:, 3:6]], 0).contiguous()
    tgt = torch.rand(N, 3, device=dev, generator=g)
    for _ in range(a.warmup):
        step_rays(rays, tgt)
        step_pose(px, tgt)
    torch.cuda.synchronize()
    t_rays, t_pose = [], []
    for _ in range(a.steps):       # alternating: both see the same host / clock conditions
        t_rays.append(event_ms(lambda: step_rays(rays, tgt)))
        t_pose.append(event_ms(lambda: step_pose(px, tgt)))

    # the pose module alone: CameraPoses forward + backward (the torch ops the graphed step captures for it), eager
    def pose_module():
        cam.se3.grad = None
        (cam() * init).sum().backward()
    for _ in range(a.warmup):
        pose_module()
    t_mod = [event_ms(pose_module) for _ in range(a.steps)]

    # the pose module's share of the graphed step: CameraPoses forward + backward (fixed upstream gradient) + the pose FusedAdam,
    # captured alone as one CUDA graph and replayed (100 replays per timed sample)
    cam2 = CameraPoses(init)
    popt2 = FusedAdam(cam2.parameters(), lr=1e-3)
    g_stack = torch.randn(V, 3, 4, device=dev, generator=g)

    def pose_part():
        popt2.zero_grad(set_to_none=True)
        cam2().backward(g_stack)
        popt2.step_captured()
    popt2.graph_begin(dev)
    popt2.graph_set_lr()
    side = torch.cuda.Stream(device=dev)
    side.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(side):
        for _ in range(3):
            pose_part()
    torch.cuda.current_stream(dev).wait_stream(side)
    torch.cuda.synchronize()
    pg = torch.cuda.CUDAGraph()
    with torch.cuda.graph(pg):
        pose_part()

    def replays():
        for _ in range(100):
            pg.replay()
    replays()
    t_mod_graph = [event_ms(replays) / 100 for _ in range(a.steps)]

    # per-call times of the new kernels at the step's shapes
    g_out = torch.randn(N, 11, device=dev, generator=g)
    ops.kernel_timer.enable(True)
    for _ in range(a.steps):
        ops.rays_from_poses(H, W, focal, init, px, near, far)
        ops.rays_from_poses_backward(init, px, H, W, focal, g_out)
    kt = {k: stats(v) for k, v in ops.kernel_timer.collect().items()}
    ops.kernel_timer.enable(False)

    r, p = stats(t_rays), stats(t_pose)
    res = {"card": card(), "cfg": "cfg 2: 4,096 rays, 64 + 64 samples, perturb 1, raw_noise_std 1, %d x %d" % (H, W),
           "views": V, "graphed_step_rays": r, "graphed_step_pose_table": p,
           "pose_table_overhead_ms": p["median_ms"] - r["median_ms"],
           "pose_module_eager_fwd_bwd": stats(t_mod), "pose_module_and_adam_graphed": stats(t_mod_graph), "kernels": kt}
    print(json.dumps(res, indent=1))
    if a.out:
        doc = json.load(open(a.out)) if os.path.isfile(a.out) else {}
        doc["timing"] = res
        with open(a.out, "w") as f:
            json.dump(doc, f, indent=1)


if __name__ == "__main__":
    main()
