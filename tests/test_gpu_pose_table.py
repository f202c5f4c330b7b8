"""Pose-table refinement on the GPU: the rays of a table of poses at given pixels (mvip_rays_from_poses) and their pose gradient,
render(c2w=stack, pixels=...) / render_deferred against float64 autograd of the reference port, GraphedTrainStep(poses=...)
against the eager loop, and pose refinement of several views against the frozen trained networks."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import torch_cpu_port as port
from test_gpu_pose_grad import ASM_REL, E2E_BARS, _cos_rel, _kwargs, _net, _params_np, _trained

pytestmark = pytest.mark.gpu

DEV = "cuda"
HERE = os.path.dirname(os.path.abspath(__file__))
FRAC = {}


def _rot(axis, deg, dtype=torch.float32):
    from mvip_nerf_b200.cameras import so3_exp
    a = torch.tensor(axis, dtype=torch.float64)
    return so3_exp(a / a.norm() * np.deg2rad(deg)).to(dtype)


def _stack_around(c2w, V, spread_deg, shift, seed):
    """V poses around c2w [3,4]: rotated by up to spread_deg about random axes (world side), centres moved by up to `shift`"""
    g = torch.Generator().manual_seed(seed)
    out = []
    for v in range(V):
        R = _rot(torch.randn(3, generator=g).tolist(), spread_deg * float(torch.rand(1, generator=g)), c2w.dtype)
        t = c2w[:, 3] + shift * (torch.rand(3, generator=g, dtype=c2w.dtype) * 2 - 1)
        out.append(torch.cat([R @ c2w[:, :3], t[:, None]], 1))
    return torch.stack(out, 0)


def _all_pixels(V, H, W, seed):
    v, i, j = torch.meshgrid(torch.arange(V), torch.arange(H), torch.arange(W), indexing="ij")
    px = torch.stack([v.reshape(-1), i.reshape(-1), j.reshape(-1)], 1)
    return px[torch.randperm(px.shape[0], generator=torch.Generator().manual_seed(seed))].to(torch.int32)


def _gd():
    return np.load(os.path.join(HERE, "golden", "ray_batch.npz"))


def _case(gd, c):
    H, W, focal, near, far, ndc, use_vd, i0, j0, h, w = gd[c + "_args"]
    return int(H), int(W), float(focal), float(near), float(far), bool(ndc), bool(use_vd), (int(i0), int(j0), int(h), int(w))


# cases of ray_batch.npz without a static camera (the pose-table entry has none)
CASES = ["plain", "ndc", "ndc_patch", "ndc_nodirs", "patch"]


# ---------------------------------------------------------------------------------------------------------------------------
# forward: bitwise equal to mvip_rays_from_pose of the matching view
# ---------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", CASES)
def test_forward_bitwise(case):
    from mvip_nerf_b200 import ops
    gd = _gd()
    H, W, focal, near, far, ndc, use_vd, win = _case(gd, case)
    c2w = torch.from_numpy(gd[case + "_c2w"]).float()
    poses = _stack_around(c2w, 3, 10.0, 0.3, CASES.index(case)).to(DEV)
    poses[0] = c2w.to(DEV)                              # view 0 is the golden pose itself
    px = _all_pixels(3, H, W, 1).to(DEV)
    got = ops.rays_from_poses(H, W, focal, poses, px, near, far, use_viewdirs=use_vd, ndc=ndc)
    full = torch.stack([ops.rays_from_pose(H, W, focal, poses[v], near, far, use_viewdirs=use_vd, ndc=ndc) for v in range(3)], 0)
    want = full[px[:, 0].long(), (px[:, 1] * W + px[:, 2]).long()]
    assert torch.equal(got.view(torch.int32), want.view(torch.int32))
    # the golden batch of view 0 over its window, in window order
    i0, j0, h, w = win
    ii, jj = torch.meshgrid(torch.arange(i0, i0 + h), torch.arange(j0, j0 + w), indexing="ij")
    wpx = torch.stack([torch.zeros_like(ii), ii, jj], -1).reshape(-1, 3).to(torch.int32).to(DEV)
    gw = ops.rays_from_poses(H, W, focal, poses[:1], wpx, near, far, use_viewdirs=use_vd, ndc=ndc)
    assert torch.equal(gw.view(torch.int32), ops.rays_from_pose(H, W, focal, c2w.to(DEV), near, far, use_viewdirs=use_vd, patch=win,
                                                                ndc=ndc).view(torch.int32))
    assert torch.equal(gw.cpu(), torch.from_numpy(gd[case + "_batch"]))
    # int64 pixels give the same rows
    assert torch.equal(ops.rays_from_poses(H, W, focal, poses, px.long(), near, far, use_viewdirs=use_vd, ndc=ndc), got)


def test_forward_out_of_range_entries_give_nan_rows():
    from mvip_nerf_b200 import ops
    H, W, focal = 20, 30, 25.0
    poses = _stack_around(torch.eye(4)[:3], 2, 5.0, 0.1, 0).to(DEV)
    px = _all_pixels(2, H, W, 2)[:64].clone()
    bad = [(-1, 0, 0), (2, 0, 0), (0, -1, 3), (0, H, 3), (1, 2, -1), (1, 2, W), (2 ** 31 - 1, 0, 0), (0, 0, -2 ** 31)]
    rows = list(range(3, 3 + 7 * len(bad), 7))
    for r, b in zip(rows, bad):
        px[r] = torch.tensor(b, dtype=torch.int32)
    px = px.to(DEV)
    for use_vd, ndc in ((True, False), (False, True)):
        got = ops.rays_from_poses(H, W, focal, poses, px, 1., 5., use_viewdirs=use_vd, ndc=ndc)
        ok = torch.ones(64, dtype=torch.bool)
        ok[rows] = False
        assert torch.isnan(got[~ok.to(DEV)]).all()
        assert torch.isfinite(got[ok.to(DEV)]).all()
        good = px[ok.to(DEV)]
        assert torch.equal(got[ok.to(DEV)], ops.rays_from_poses(H, W, focal, poses, good, 1., 5., use_viewdirs=use_vd, ndc=ndc))
    # int64 values beyond int32 stay out of range
    big = torch.tensor([[2 ** 32, 0, 0], [0, 0, 2 ** 32 + 1]], device=DEV)
    assert torch.isnan(ops.rays_from_poses(H, W, focal, poses, big, 1., 5.)).all()


# ---------------------------------------------------------------------------------------------------------------------------
# backward: d poses against float64 autograd of one pose copy per pixel
# ---------------------------------------------------------------------------------------------------------------------------
def _batch64(H, W, focal, near, far, ndc, use_vd, px, pose_pp):
    """the batch render() assembles (run.py:1171-1207) in float64 for pixels px [n,3] with one pose per pixel [n,3,4]"""
    from mvip_nerf_b200.run_nerf_helpers import ndc_rays
    i, j = px[:, 1].double(), px[:, 2].double()
    dirs = torch.stack([(j - W * .5) / focal, -(i - H * .5) / focal, -torch.ones_like(i)], -1)
    rd = (dirs[:, None, :] * pose_pp[:, :3, :3]).sum(-1)
    ro = pose_pp[:, :3, 3]
    vd = rd / torch.norm(rd, dim=-1, keepdim=True)
    if ndc:
        ro, rd = ndc_rays(H, W, focal, 1., ro, rd)
    ones = torch.ones_like(rd[:, :1])
    return torch.cat([ro, rd, near * ones, far * ones] + ([vd] if use_vd else []), -1)


BWD_CASES = [(case, V) for case in ("plain", "ndc", "ndc_nodirs") for V in (1, 3, 20)]


@pytest.mark.parametrize("case,V", BWD_CASES)
def test_backward_vs_float64(case, V):
    from mvip_nerf_b200 import ops
    gd = _gd()
    H, W, focal, near, far, ndc, use_vd, _ = _case(gd, case)
    c2w = torch.from_numpy(gd[case + "_c2w"]).float()
    poses = _stack_around(c2w, V, 10.0, 0.3, V)
    g = torch.Generator().manual_seed(V * 10 + CASES.index(case))
    used = torch.arange(V) if V <= 3 else torch.randperm(V, generator=g)[:V - 5]      # V = 20: five views get no ray
    n = 3000 if V > 1 else H * W
    px = torch.stack([used[torch.randint(len(used), (n,), generator=g)], torch.randint(H, (n,), generator=g),
                      torch.randint(W, (n,), generator=g)], 1).to(torch.int32)
    stride = 11 if use_vd else 8
    g_out = torch.randn(n, stride, generator=g, dtype=torch.float64)
    pp = poses.double()[px[:, 0].long()].clone().requires_grad_(True)
    term = torch.autograd.grad((_batch64(H, W, focal, near, far, ndc, use_vd, px, pp) * g_out).sum(), [pp])[0]
    want = torch.zeros(V, 3, 4, dtype=torch.float64).index_add_(0, px[:, 0].long(), term)
    bar = ASM_REL * torch.zeros(V, 3, 4, dtype=torch.float64).index_add_(0, px[:, 0].long(), term.abs())
    got = ops.rays_from_poses_backward(poses.to(DEV), px.to(DEV), H, W, focal, g_out.float().to(DEV), use_viewdirs=use_vd, ndc=ndc)
    err = (got.cpu().double() - want).abs()
    unused = torch.ones(V, dtype=torch.bool)
    unused[used] = False
    assert torch.equal(got[unused.to(DEV)], torch.zeros_like(got[unused.to(DEV)]))
    frac = float((err / bar.clamp_min(1e-300))[~unused].max())
    FRAC.setdefault("backward", []).append([case, V, frac])
    assert (err <= bar).all(), frac
    # bitwise reproducible
    assert torch.equal(got, ops.rays_from_poses_backward(poses.to(DEV), px.to(DEV), H, W, focal, g_out.float().to(DEV),
                                                         use_viewdirs=use_vd, ndc=ndc))
    if V == 1:     # the whole image in shuffled order agrees with the single-pose entry within the same bar
        full = _all_pixels(1, H, W, 5)
        gf = torch.zeros(H * W, stride, dtype=torch.float64)
        gf[(full[:, 1] * W + full[:, 2]).long()] = torch.randn(H * W, stride, generator=g, dtype=torch.float64)
        g_pix = gf[(full[:, 1] * W + full[:, 2]).long()]
        a = ops.rays_from_poses_backward(poses.to(DEV), full.to(DEV), H, W, focal, g_pix.float().to(DEV), use_viewdirs=use_vd, ndc=ndc)
        b, _ = ops.rays_from_pose_backward(poses[0].to(DEV), None, H, W, focal, (0, 0, H, W), gf.float().to(DEV),
                                           use_viewdirs=use_vd, ndc=ndc)
        pp = poses.double()[full[:, 0].long()].clone().requires_grad_(True)
        t1 = torch.autograd.grad((_batch64(H, W, focal, near, far, ndc, use_vd, full, pp) * g_pix).sum(), [pp])[0]
        bar1 = ASM_REL * t1.abs().sum(0)
        d = (a[0] - b).abs().cpu().double()
        FRAC.setdefault("single_pose_entry", []).append([case, float((d / bar1.clamp_min(1e-300)).max())])
        assert (d <= bar1).all()


def test_backward_ignores_out_of_range_entries():
    from mvip_nerf_b200 import ops
    H, W, focal = 16, 24, 20.0
    poses = _stack_around(torch.eye(4)[:3], 3, 5.0, 0.1, 1).to(DEV)
    px = _all_pixels(3, H, W, 3)[:500].to(DEV)
    g = torch.randn(500, 11, device=DEV, generator=torch.Generator(device=DEV).manual_seed(1))
    ref = ops.rays_from_poses_backward(poses, px, H, W, focal, g)
    bad = torch.tensor([[-1, 0, 0], [3, 1, 1], [0, H, 0], [1, 0, W], [2, -1, 2]], dtype=torch.int32, device=DEV)
    px2 = torch.cat([px[:200], bad, px[200:]], 0)
    g2 = torch.cat([g[:200], torch.full((5, 11), 1e30, device=DEV), g[200:]], 0)
    got = ops.rays_from_poses_backward(poses, px2, H, W, focal, g2)
    # the valid entries' chunk positions moved, so the summation order did too: equal within fp32 summation order
    assert torch.isfinite(got).all()
    torch.testing.assert_close(got, ref, rtol=1e-5, atol=1e-5)


# ---------------------------------------------------------------------------------------------------------------------------
# end to end: render(c2w=stack, pixels=...) d stack against float64 autograd of the reference port
# ---------------------------------------------------------------------------------------------------------------------------
# (min cos, max rel-L2): the c2w bars of test_gpu_pose_grad.E2E_BARS (one 16 x 16 patch of one pose) widened to about 1.5x the
# deviation measured here on a B200 (1000 W) for 768 pixels of three poses: random cos 0.9954 / rel 0.097, trained 0.9830 / 0.185
PIXELS_E2E_BARS = {"random": (min(E2E_BARS[("random", "c2w", "c2w")][0], 0.993), max(E2E_BARS[("random", "c2w", "c2w")][1], 0.145)),
                   "trained": (min(E2E_BARS[("trained", "c2w", "c2w")][0], 0.974), max(E2E_BARS[("trained", "c2w", "c2w")][1], 0.28))}


@pytest.mark.parametrize("which", ["random", "trained"])
def test_render_pixels_grad_vs_reference(which):
    from mvip_nerf_b200.run import render, render_deferred
    if which == "trained":
        d, (nc, nf) = _trained()
        H, W, focal, near, far = int(d["H"]), int(d["W"]), float(d["focal"]), float(d["near"]), float(d["far"])
        c2w0 = torch.from_numpy(d["c2w"]).double()
    else:
        nc, nf = _net(11), _net(12)
        H, W, focal, near, far = 64, 80, 70.0, 2.0, 6.0
        c2w0 = torch.tensor([[1, 0, 0, 0.1], [0, 1, 0, -0.2], [0, 0, 1, 4.0]], dtype=torch.float64)
    for net in (nc, nf):
        for p in net.parameters():
            p.requires_grad_(False)
    kw = _kwargs(nc, nf)
    V = 3
    stack = _stack_around(c2w0.float(), V, 1.0, 0.01 * (far - near), 9).double()
    g = torch.Generator().manual_seed(3)
    n = 768
    px = torch.stack([torch.randint(V, (n,), generator=g), H // 4 + torch.randint(H // 2, (n,), generator=g),
                      W // 4 + torch.randint(W // 2, (n,), generator=g)], 1).to(torch.int32)
    g_rgb = torch.randn(n, 3, generator=g, dtype=torch.float64)
    leaf = stack.clone().requires_grad_(True)
    b64 = _batch64(H, W, focal, near, far, False, True, px, leaf[px[:, 0].long()])
    pc = {k: v.double() for k, v in port.params_from_numpy(_params_np(nc)).items()}
    pf = {k: v.double() for k, v in port.params_from_numpy(_params_np(nf)).items()}
    out = port.render_rays(b64, pc, pf, torch.linspace(0., 1., 64, dtype=torch.float64), lindisp=True, white_bkgd=True)
    with torch.no_grad():     # ill-conditioned rays (reference density at the last sample within 5e-3 of zero): no upstream grad
        pts = b64[:, None, 0:3] + b64[:, None, 3:6] * out["z_vals"][..., None]
        keep = (port.query(pf, pts, b64[:, -3:])[:, -1, 3].abs() > 5e-3).double()[:, None]
    want = torch.autograd.grad((out["rgb_map"] * g_rgb * keep).sum(), [leaf])[0]
    res = {}
    for name, fn in (("render", render), ("render_deferred", render_deferred)):
        x = stack.float().to(DEV).requires_grad_(True)
        rgb, _, _, _, _ = fn(H, W, focal, c2w=x, pixels=px.to(DEV), near=near, far=far, **kw)
        assert rgb.shape == (n, 3)
        (rgb.double() * (g_rgb * keep).to(DEV)).sum().backward()
        res[name] = x.grad.clone()
    assert torch.equal(res["render"], res["render_deferred"])
    got = res["render"].double().cpu()
    assert torch.isfinite(got).all()
    cos, rel = _cos_rel(got, want)
    FRAC.setdefault("e2e", []).append([which, int(keep.sum()), cos, rel])
    min_cos, max_rel = PIXELS_E2E_BARS[which]
    assert cos > min_cos and rel < max_rel, (cos, rel)


def test_no_grad_stack_runs_forward_kernel_only():
    from mvip_nerf_b200 import ops
    from mvip_nerf_b200.run import render
    nc, nf = _net(21), _net(22)
    kw = _kwargs(nc, nf)
    stack = _stack_around(torch.tensor([[1., 0, 0, 0.1], [0, 1, 0, -0.2], [0, 0, 1, 4.0]]), 4, 2.0, 0.1, 2).to(DEV)
    px = _all_pixels(4, 48, 64, 4)[:2048].to(DEV)
    calls = []
    real = ops._call
    ops._call = lambda name, *a: (calls.append(name if isinstance(name, str) else name[0]), real(name, *a))[1]
    try:
        rgb, *_ = render(48, 64, 60.0, c2w=stack, pixels=px, near=2., far=6., **kw)
        rgb.sum().backward()
    finally:
        ops._call = real
    assert "mvip_rays_from_poses" in calls and "mvip_rays_from_poses_backward" not in calls
    # the pixels= batch equals the rays= batch of the same rays (the same kernels downstream)
    rays_flat = ops.rays_from_poses(48, 64, 60.0, stack, px, 2., 6.)
    rgb2, *_ = render(48, 64, 60.0, rays=(rays_flat[:, 0:3], rays_flat[:, 3:6]), near=2., far=6., **kw)
    assert torch.equal(rgb.detach(), rgb2.detach())


# ---------------------------------------------------------------------------------------------------------------------------
# GraphedTrainStep(poses=...) == the eager loop
# ---------------------------------------------------------------------------------------------------------------------------
def test_graphed_pose_step_matches_eager():
    from mvip_nerf_b200 import run
    from mvip_nerf_b200.cameras import CameraPoses
    from mvip_nerf_b200.graph import GraphedTrainStep, default_loss
    from mvip_nerf_b200.optim import FusedAdam
    H, W, focal, near, far = 64, 80, 70.0, 2.0, 6.0
    V, N, steps = 5, 2048, 5
    init = _stack_around(torch.tensor([[1., 0, 0, 0.1], [0, 1, 0, -0.2], [0, 0, 1, 4.0]]), V, 3.0, 0.1, 6).to(DEV)
    g = torch.Generator().manual_seed(8)
    pxs = [torch.stack([torch.randint(V, (N,), generator=g), torch.randint(H, (N,), generator=g), torch.randint(W, (N,), generator=g)],
                       1).to(torch.int32).to(DEV) for _ in range(steps)]
    tgts = [torch.rand(N, 3, generator=g).to(DEV) for _ in range(steps)]

    def setup():      # the networks of the random end-to-end case: they have density along these rays, so d stack != 0
        nc, nf = _net(11), _net(12)
        kw = _kwargs(nc, nf)
        params = [p for net in (nc, nf) for p in net.parameters()]
        cam = CameraPoses(init)
        return kw, (nc, nf), params, cam, FusedAdam(params, lr=5e-4), FusedAdam(cam.parameters(), lr=1e-3)

    kw, nets, params_a, cam_a, opt_a, popt_a = setup()
    losses_a = []
    for px, tgt in zip(pxs, tgts):
        opt_a.zero_grad(set_to_none=True)
        popt_a.zero_grad(set_to_none=True)
        out = run.render(H, W, focal, chunk=32768, c2w=cam_a(), pixels=px, near=near, far=far, _mse=(tgt, None), **kw)
        loss = default_loss(*out, tgt, 1.0)
        loss.backward()
        opt_a.step()
        popt_a.step()
        for net in nets:
            net.repack()
        losses_a.append(loss.detach().clone())

    kw, nets, params_b, cam_b, opt_b, popt_b = setup()
    before = [p.detach().clone() for p in params_b + [cam_b.se3]]
    step = GraphedTrainStep(kw, opt_b, H, W, focal, N, near, far, poses=cam_b, pose_optimizer=popt_b)
    assert step.fused_loss
    step.pixels.copy_(pxs[0])
    step.target.copy_(tgts[0])
    step.capture()
    assert all(torch.equal(a, b) for a, b in zip(before, params_b + [cam_b.se3]))          # capture trains nothing
    assert float(popt_b.state[cam_b.se3]["exp_avg"].abs().max()) == 0.0
    losses_b = [step(px, tgt).clone() for px, tgt in zip(pxs, tgts)]
    dl = max(float((a - b).abs()) for a, b in zip(losses_a, losses_b))
    dp = max(float((a - b).detach().abs().max()) for a, b in zip(params_a, params_b))
    ds = float((cam_a.se3 - cam_b.se3).detach().abs().max())
    FRAC["graphed_vs_eager"] = {"loss": dl, "params": dp, "se3": ds, "se3_max": float(cam_a.se3.detach().abs().max())}
    assert float(cam_a.se3.abs().max()) > 0
    assert all(torch.equal(a, b) for a, b in zip(losses_a, losses_b)), dl
    assert all(torch.equal(a, b) for a, b in zip(params_a, params_b)), dp
    assert torch.equal(cam_a.se3, cam_b.se3), ds
    assert float(popt_b.state_dict()["state"][0]["step"]) == steps


# ---------------------------------------------------------------------------------------------------------------------------
# refinement of six views against the frozen trained networks, and a joint run
# ---------------------------------------------------------------------------------------------------------------------------
def _refine_setup():
    from mvip_nerf_b200.run import render
    d, (nc, nf) = _trained()
    for net in (nc, nf):
        for p in net.parameters():
            p.requires_grad_(False)
    f = 4
    H, W, focal, near, far = int(d["H"]) // f, int(d["W"]) // f, float(d["focal"]) / f, float(d["near"]), float(d["far"])
    kw = _kwargs(nc, nf)
    c2w = torch.from_numpy(d["c2w"]).float()
    V = 6
    true = _stack_around(c2w, V, 1.5, 0.02 * (far - near), 11).to(DEV)
    with torch.no_grad():
        imgs = torch.stack([render(H, W, focal, c2w=true[v], near=near, far=far, **kw)[0] for v in range(V)], 0)
    g = torch.Generator().manual_seed(12)
    start = []
    for v in range(V):      # 1 degree about a random axis, 1 % of the depth range in a random direction
        dt = torch.randn(3, generator=g)
        start.append(torch.cat([_rot(torch.randn(3, generator=g).tolist(), 1.0).to(DEV) @ true[v, :, :3],
                                (true[v, :, 3] + (dt / dt.norm() * 0.01 * (far - near)).to(DEV))[:, None]], 1))
    return kw, (nc, nf), (H, W, focal, near, far), true, imgs, torch.stack(start, 0)


def _pose_errs(est, true):
    Rrel = est[:, :, :3] @ true[:, :, :3].transpose(1, 2)
    tr = Rrel.diagonal(dim1=1, dim2=2).sum(-1)
    ang = torch.arccos(((tr - 1) / 2).clamp(-1, 1))
    return ang.cpu(), (est[:, :, 3] - true[:, :, 3]).norm(dim=-1).cpu()


REFINE_STEPS = 300


def fine_mse(rgb, disp, acc, depth, extras, target, scale):
    """img2mse of the fine map only: the targets are the fine network's renders at the true poses, so this loss is zero there.
    (The default loss adds img2mse(rgb0, target); the coarse map differs from the fine target even at the true poses, which
    would leave a floor whose pose gradient pulls the optimum away from them.)"""
    from mvip_nerf_b200.run_nerf_helpers import img2mse
    return img2mse(rgb, target) * scale


def test_refinement_converges():
    from mvip_nerf_b200.cameras import CameraPoses
    from mvip_nerf_b200.graph import GraphedTrainStep
    from mvip_nerf_b200.optim import FusedAdam
    kw, _, (H, W, focal, near, far), true, imgs, start = _refine_setup()
    V, N = true.shape[0], 4096
    cam = CameraPoses(start)
    lr0 = 1e-2
    popt = FusedAdam(cam.parameters(), lr=lr0)
    step = GraphedTrainStep(kw, None, H, W, focal, N, near, far, loss_fn=fine_mse, poses=cam, pose_optimizer=popt)
    g = torch.Generator(device=DEV).manual_seed(13)
    a0, t0 = _pose_errs(cam().detach(), true)
    losses = []
    for it in range(REFINE_STEPS):
        px = torch.stack([torch.randint(V, (N,), device=DEV, generator=g), torch.randint(H, (N,), device=DEV, generator=g),
                          torch.randint(W, (N,), device=DEV, generator=g)], 1).to(torch.int32)
        tgt = imgs[px[:, 0].long(), px[:, 1].long(), px[:, 2].long()]
        popt.param_groups[0]["lr"] = lr0 * 0.5 * (1 + np.cos(np.pi * it / REFINE_STEPS))
        losses.append(float(step(px, tgt)))
    a1, t1 = _pose_errs(cam().detach(), true)
    FRAC["refine"] = {"steps": REFINE_STEPS, "rot_ratio": (a1 / a0).tolist(), "trans_ratio": (t1 / t0).tolist(),
                      "loss_first": float(np.mean(losses[:5])), "loss_last": float(np.mean(losses[-5:]))}
    assert np.isfinite(losses).all()
    assert np.mean(losses[-5:]) <= 0.5 * np.mean(losses[:5])
    assert (a1 <= 0.5 * a0).all() and (t1 <= 0.5 * t0).all(), (a1 / a0, t1 / t0)


def test_joint_refinement_stays_finite_and_learns():
    from mvip_nerf_b200.cameras import CameraPoses
    from mvip_nerf_b200.graph import GraphedTrainStep
    from mvip_nerf_b200.optim import FusedAdam
    kw, nets, (H, W, focal, near, far), true, imgs, start = _refine_setup()
    params = [p for net in nets for p in net.parameters()]
    for p in params:
        p.requires_grad_(True)
    V, N = true.shape[0], 4096
    cam = CameraPoses(start)
    step = GraphedTrainStep(kw, FusedAdam(params, lr=1e-4), H, W, focal, N, near, far, poses=cam,
                            pose_optimizer=FusedAdam(cam.parameters(), lr=1e-3))
    g = torch.Generator(device=DEV).manual_seed(14)
    losses = []
    for _ in range(60):
        px = torch.stack([torch.randint(V, (N,), device=DEV, generator=g), torch.randint(H, (N,), device=DEV, generator=g),
                          torch.randint(W, (N,), device=DEV, generator=g)], 1).to(torch.int32)
        losses.append(float(step(px, imgs[px[:, 0].long(), px[:, 1].long(), px[:, 2].long()])))
    FRAC["joint"] = {"loss_first": float(np.mean(losses[:5])), "loss_last": float(np.mean(losses[-5:]))}
    assert np.isfinite(losses).all() and all(torch.isfinite(p).all() for p in params + [cam.se3])
    assert np.mean(losses[-5:]) < np.mean(losses[:5])


def test_record_fractions():
    """merges the measured fractions of the bars into the JSON file named by MVIP_POSE_TABLE_OUT (key "bars")"""
    out = os.environ.get("MVIP_POSE_TABLE_OUT")
    if out:
        doc = json.load(open(out)) if os.path.isfile(out) else {}
        doc["bars"] = FRAC
        with open(out, "w") as f:
            json.dump(doc, f, indent=1)
