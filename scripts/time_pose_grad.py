"""Times the pose / ray gradient path on one GPU and prints one JSON document (card name and power limit included).

  * cfg 2: 4,096 rays, 64 + 128 samples, eager render + backward, with and without c2w.requires_grad (CUDA events, median);
  * one 512 x 512 guidance view through render_deferred with a pose gradient;
  * per-kernel times of the new entries (ops.kernel_timer) and the input-gradient kernel's achieved bandwidth against the
    6,545 GB/s copy peak, timed in points mode: its algorithmic bytes are 1,280 B per point of dZ read, 24 B per point of inputs
    read (pts, dirs) and 24 B per point written.

usage: python scripts/time_pose_grad.py [--out FILE] [--iters N]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

COPY_PEAK_GBS = 6545.0


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else torch.cuda.get_device_name()


def kwargs(nc, nf, n_fine):
    from mvip_nerf_b200.run import _FusedQuery
    from mvip_nerf_b200.run_nerf_helpers import get_embedder
    e, _ = get_embedder(10)
    ev, _ = get_embedder(4)
    return dict(network_query_fn=_FusedQuery(e, ev, 65536), network_fn=nc, network_fine=nf, N_samples=64, N_importance=n_fine,
                perturb=1., raw_noise_std=1., white_bkgd=False, lindisp=False, use_viewdirs=True, ndc=False)


def timed(fn, iters):
    for _ in range(3):
        fn()
    ts = []
    for _ in range(iters):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    ts.sort()
    return ts[len(ts) // 2]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--iters", type=int, default=20)
    a = ap.parse_args()
    from mvip_nerf_b200 import ops
    from mvip_nerf_b200.run import render, render_deferred
    from mvip_nerf_b200.run_nerf_helpers import NeRF
    dev = torch.device("cuda")
    torch.manual_seed(0)
    nc = NeRF(input_ch=63, input_ch_views=27, use_viewdirs=True).to(dev)
    nf = NeRF(input_ch=63, input_ch_views=27, use_viewdirs=True).to(dev)
    res = {"card": card()}
    # cfg 2: 4,096 rays as a 64 x 64 patch of a 756 x 1008 view
    H, W, focal = 756, 1008, 767.2935
    c2w0 = torch.tensor([[1, 0, 0, 0.], [0, 1, 0, 0.], [0, 0, 1, 0.]], device=dev)
    kw = kwargs(nc, nf, 128)

    def step(pose_grad):
        c = c2w0.clone().requires_grad_(pose_grad)
        rgb, disp, acc, depth, ex = render(H, W, focal, chunk=1 << 15, c2w=c, near=2., far=6., patch=(346, 472, 64, 64), **kw)
        (rgb.square().mean() + ex["rgb0"].square().mean()).backward()
    for k in ("cfg2_render_backward_ms", "cfg2_render_backward_pose_grad_ms"):
        res[k] = timed(lambda: step(k.endswith("pose_grad_ms")), a.iters)
    ops.kernel_timer.enable(True)
    step(True)
    ops.kernel_timer.collect()
    ops.kernel_timer.enable(True)
    for _ in range(a.iters):
        step(True)
    rec = ops.kernel_timer.collect()
    ops.kernel_timer.enable(False)
    per = {k: sorted(v)[len(v) // 2] for k, v in rec.items()}
    res["cfg2_per_call_median_ms"] = per
    # the input-gradient launch of the fine pass: 4,096 x 192 points; bracketed separately in points mode for a clean kernel time
    P = 4096 * 192
    pts = torch.randn(P, 3, device=dev)
    dirs = torch.nn.functional.normalize(torch.randn(P, 3, device=dev), dim=-1)
    packed = nf.packed()
    raw, stash = ops.mlp_forward(packed, pts=pts, dirs=dirs, want_stash=True)
    _, ws = ops.mlp_backward(packed, torch.randn_like(raw) * 1e-2, stash, want_workspace=True)
    del stash
    ms = timed(lambda: ops.mlp_input_grad(packed, ws, pts=pts, dirs=dirs), max(a.iters, 50))
    nbytes = P * (1280 + 24 + 24)          # dZ read, pts + dirs read, d pts + d dirs written
    res["input_grad_points"] = {"points": P, "ms": ms, "GB_per_s": nbytes / ms / 1e6,
                                "frac_of_copy_peak": nbytes / ms / 1e6 / COPY_PEAK_GBS}
    del ws
    # one 512 x 512 guidance view, deferred backward, pose gradient
    kw64 = kwargs(nc, nf, 64)

    def guide():
        c = c2w0.clone().requires_grad_(True)
        rgb, disp, acc, depth, ex = render_deferred(512, 512, 443.4, chunk=1 << 13, c2w=c, near=2., far=6., **kw64)
        rgb.square().mean().backward()
    res["guidance_512_deferred_pose_grad_ms"] = timed(guide, 3)
    res["peak_mem_GB"] = torch.cuda.max_memory_allocated() / 1e9
    txt = json.dumps(res, indent=1)
    print(txt)
    if a.out:
        with open(a.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
