"""Gradients of render() with respect to rays and camera poses: the MLP input gradient (mlp_input_grad_kernel), the compositing
d |rays_d| (mvip_composite_backward_rays), the ray-assembly backward (mvip_rays_pack_backward / mvip_rays_from_pose_backward) and
their use through render() / render_deferred()."""
import numpy as np
import pytest
import torch

import mlp_ref64 as R
from oracle import torch_cpu_port as port

pytestmark = pytest.mark.gpu

DEV = "cuda"


def _net(seed):
    from mvip_nerf_b200.run_nerf_helpers import NeRF
    torch.manual_seed(seed)
    return NeRF(input_ch=63, input_ch_views=27, use_viewdirs=True).to(DEV)


def _params_np(net):
    return {k: v.detach().cpu().numpy() for k, v in net.named_parameters()}


# ---------------------------------------------------------------------------------------------------------------------------
# 1. input gradient of the fused MLP, teacher-forced from the kernel's own dZ images, every tile
# ---------------------------------------------------------------------------------------------------------------------------
def _pe_chain64(x, dpe, L, accbar):
    """float64 d x [P,3] from d PE [P, 3 + 6L] and its bar.

    Bar, derived: each d PE element is an fp32 sum over K products of bf16 operands, off by at most ACC_FLOOR * sum |dZ||W|
    (accbar, the floor mlp_ref64 uses for every MMA output).  The chain multiplies element (k, sin|cos) by 2^k cos|sin, so that
    error enters with weight 2^k.  The kernel's sin / cos of 2^k x come from pe_axis: the phase in turns is exact to ~2^-24 of
    |2^k x / 2 pi| and sin.approx adds ~2^-21, so |sin err| <= 2^-21 + 2^k |x| 2^-24; it multiplies |d PE| of the other column.
    The fp32 accumulation of the 1 + 2L terms adds (1 + 2L) 2^-24 of their absolute sum; 4x margin on the whole."""
    out = dpe[:, 0:3].clone()
    bar = accbar[:, 0:3].clone()
    absum = dpe[:, 0:3].abs()
    for k in range(L):
        f = 2.0 ** k
        s, c = torch.sin(f * x), torch.cos(f * x)
        ds, dc = dpe[:, 3 + 6 * k:6 + 6 * k], dpe[:, 6 + 6 * k:9 + 6 * k]
        term = f * (c * ds - s * dc)
        out += term
        absum += term.abs()
        esc = 2.0 ** -21 + f * x.abs() * 2.0 ** -24
        bar += f * (accbar[:, 3 + 6 * k:6 + 6 * k] + accbar[:, 6 + 6 * k:9 + 6 * k]) + f * esc * (ds.abs() + dc.abs())
    bar += (1 + 2 * L) * 2.0 ** -24 * absum
    return out, 4 * bar


def _input_grad_ref(net, ws, P, x, v):
    """float64 (d pts, bar, d view, bar) [P,3] each from the dZ images in ws"""
    p = {k: t.detach().double() for k, t in net.named_parameters()}
    W0 = R.bf16(p["pts_linears.0.weight"])
    W5 = R.bf16(p["pts_linears.5.weight"][:, :63])
    Wv = R.bf16(p["views_linears.0.weight"][:, 256:283])
    T = R.num_tiles(P)
    img = R._images(ws, R.DZ_TILE_BYTES, 38, range(0, T))
    dz0, dz5, dh = R._cols(img, 34, 38)[:P], R._cols(img, 14, 18)[:P], R._cols(img, 0, 2)[:P]
    dpe = dz0 @ W0 + dz5 @ W5
    acc = R.ACC_FLOOR * (dz0.abs() @ W0.abs() + dz5.abs() @ W5.abs())
    dpv = dh @ Wv
    accv = R.ACC_FLOOR * (dh.abs() @ Wv.abs())
    dx, bx = _pe_chain64(x.double(), dpe, 10, acc)
    dv, bv = _pe_chain64(v.double(), dpv, 4, accv)
    return dx, bx, dv, bv


def _run_backward(net, **kw):
    from mvip_nerf_b200 import ops
    packed = net.packed()
    raw, stash = ops.mlp_forward(packed, want_stash=True, **kw)
    g = torch.Generator(device=DEV).manual_seed(7)
    d_raw = torch.randn(raw.shape, device=DEV, generator=g) * 1e-2
    _, ws = ops.mlp_backward(packed, d_raw, stash, want_workspace=True)
    return packed, ws


FRAC = []


@pytest.mark.parametrize("P", [1, 127, 128, 129, 148 * 128 * 2 + 5])
def test_input_grad_points(P):
    from mvip_nerf_b200 import ops
    net = _net(1)
    g = torch.Generator(device=DEV).manual_seed(P)
    pts = torch.randn(P, 3, device=DEV, generator=g)
    dirs = torch.nn.functional.normalize(torch.randn(P, 3, device=DEV, generator=g), dim=-1)
    packed, ws = _run_backward(net, pts=pts, dirs=dirs)
    dp, dd = ops.mlp_input_grad(packed, ws, pts=pts, dirs=dirs)
    dx, bx, dv, bv = _input_grad_ref(net, ws, P, pts, dirs)
    assert torch.isfinite(dp).all() and torch.isfinite(dd).all()
    ex, ev = (dp.double() - dx).abs(), (dd.double() - dv).abs()
    assert (ex <= bx).all(), float((ex / bx).max())
    assert (ev <= bv).all(), float((ev / bv).max())
    FRAC.append(("points", P, float((ex / bx).max()), float((ev / bv).max())))
    # bitwise reproducible
    dp2, dd2 = ops.mlp_input_grad(packed, ws, pts=pts, dirs=dirs)
    assert torch.equal(dp, dp2) and torch.equal(dd, dd2)


@pytest.mark.parametrize("N,S", [(1, 64), (3, 96), (4096, 64), (4096, 128), (37, 200)])
def test_input_grad_rays(N, S):
    from mvip_nerf_b200 import ops
    net = _net(2)
    g = torch.Generator(device=DEV).manual_seed(N * 1000 + S)
    rays = torch.randn(N, 11, device=DEV, generator=g)
    rays[:, 8:11] = torch.nn.functional.normalize(rays[:, 8:11], dim=-1)
    z = torch.sort(torch.rand(N, S, device=DEV, generator=g) * 4 + 0.5, -1)[0]
    packed, ws = _run_backward(net, rays=rays, z_vals=z)
    d = ops.mlp_input_grad(packed, ws, rays=rays, z_vals=z, viewdir_offset=8)
    P = N * S
    x = rays[:, None, 0:3] + rays[:, None, 3:6] * z[..., None]            # fp32, as the kernel: o + (d * z)
    v = rays[:, None, 8:11].expand(N, S, 3).reshape(P, 3)
    dx, bx, dv, bv = _input_grad_ref(net, ws, P, x.reshape(P, 3), v)
    zz = z.double().reshape(P, 1)
    want = torch.cat([dx.view(N, S, 3).sum(1), (zz * dx).view(N, S, 3).sum(1), torch.zeros(N, 2, dtype=torch.float64, device=DEV),
                      dv.view(N, S, 3).sum(1)], 1)
    # per-point bars add up; the fixed-order fp32 sum of S terms adds S 2^-24 of their absolute sum
    sb = lambda b, t: b.view(N, S, 3).sum(1) + S * 2.0 ** -24 * t.abs().view(N, S, 3).sum(1)   # noqa: E731
    bar = torch.cat([sb(bx, dx), sb(zz.abs() * bx, zz * dx), torch.zeros(N, 2, dtype=torch.float64, device=DEV), sb(bv, dv)], 1)
    err = (d.double() - want).abs()
    assert (err <= bar).all(), float((err / bar.clamp_min(1e-30)).max())
    FRAC.append(("rays", P, float((err / bar.clamp_min(1e-30)).max()), 0.0))
    assert torch.equal(d, ops.mlp_input_grad(packed, ws, rays=rays, z_vals=z, viewdir_offset=8))


# ---------------------------------------------------------------------------------------------------------------------------
# 2. compositing: d rays_d against float64 autograd of the reference's raw2outputs (oracle.torch_cpu_port.composite)
# ---------------------------------------------------------------------------------------------------------------------------
def _composite_inputs(S, white, noisy):
    """S = 64 / 128: the raw2outputs goldens (raw, z, rays_d, noise and the upstream gradients of that case); any other S: seeded
    random inputs of the same kind (the goldens exist for 64 and 128 only)"""
    import os
    if S in (64, 128):
        fx = np.load(os.path.join(os.path.dirname(__file__), "golden", "raw2outputs.npz"))
        tag = "S%d_w%d_n%d_" % (S, white, noisy)
        t = lambda k: torch.from_numpy(fx[k].copy())   # noqa: E731
        return (t("S%d_raw" % S), t("S%d_z" % S), t("S%d_rays_d" % S), t("S%d_noise" % S) if noisy else None,
                t(tag + "g_rgb"), t(tag + "g_disp"), t(tag + "g_acc"), t(tag + "g_depth"), t(tag + "g_weights"))
    g = torch.Generator().manual_seed(1000 + S * 4 + white * 2 + noisy)
    N = 48
    r = lambda *s: torch.randn(*s, generator=g)   # noqa: E731
    return (r(N, S, 4), torch.sort(torch.rand(N, S, generator=g) * 5 + 1, -1)[0], r(N, 3), r(N, S) if noisy else None,
            r(N, 3), r(N), r(N), r(N), r(N, S))


COMPOSITE_CASES = [(S, w, n, f) for S in (64, 128) for w in (0, 1) for n in (0, 1) for f in (0, 1)] + \
                  [(45, w, n, 0) for w in (0, 1) for n in (0, 1)]


@pytest.mark.parametrize("S,white,noisy,fused", COMPOSITE_CASES)
def test_composite_rays_d(S, white, noisy, fused):
    from mvip_nerf_b200 import ops
    raw, z, rd, noise, g_rgb, g_disp, g_acc, g_depth, g_w = _composite_inputs(S, white, noisy)
    N = raw.shape[0]
    g = torch.Generator().manual_seed(S + 7)
    t_rgb, t_disp, g_sq = torch.rand(N, 3, generator=g), torch.rand(N, generator=g), torch.tensor([0.7, 0.3])
    r64, d64 = raw.double().requires_grad_(True), rd.double().requires_grad_(True)
    rgb, disp, acc, w, depth = port.composite(r64, z.double(), d64, None if noise is None else noise.double(), bool(white))
    loss = (rgb * g_rgb.double()).sum() + (disp * g_disp.double()).sum() + (acc * g_acc.double()).sum() + \
        (depth * g_depth.double()).sum() + (w * g_w.double()).sum()
    if fused:
        loss = loss + g_sq[0].double() * ((rgb - t_rgb.double()) ** 2).sum() + g_sq[1].double() * ((disp - t_disp.double()) ** 2).sum()
    want_d = torch.autograd.grad(loss, [d64])[0]
    cu = lambda t: None if t is None else t.to(DEV)   # noqa: E731
    args = (cu(raw), cu(z), cu(rd), cu(noise), white, False, cu(g_rgb), cu(g_disp), cu(g_acc), cu(g_depth), cu(g_w), None)
    fk = dict(target_rgb=cu(t_rgb), target_disp=cu(t_disp), g_sq=cu(g_sq)) if fused else {}
    d_raw, d_dir = ops.composite_backward(*args, want_rays_d=True, **fk)
    assert torch.equal(d_raw, ops.composite_backward(*args, **fk))     # d_raw does not depend on the new option
    got = d_dir.cpu().double()
    assert torch.equal(torch.isnan(got), torch.isnan(want_d))
    # A sample with 0 < sigma + noise < 1e-3 at the last position (dist 1e10) makes d |rays_d| ill-conditioned: relu(sigma) 1e10
    # e^(-sigma 1e10 |d|) swings with an ulp of sigma, in the reference as well (SURVEY section 7).  Such rays are left out of the
    # value comparison (a departure from comparing every ray); how many are left out is recorded.
    s = raw[..., 3] + (noise if noise is not None else 0)
    ok = ~((s > 0) & (s < 1e-3)).any(1) & ~torch.isnan(want_d).any(1)
    scale = want_d[ok].abs().max()
    err = float((got[ok] - want_d[ok]).abs().max() / scale)
    FRAC.append(("composite", S, white, noisy, fused, int((~ok).sum()), int(torch.isnan(want_d).any(1).sum()), err / 2e-5))
    assert err <= 2e-5, err


# ---------------------------------------------------------------------------------------------------------------------------
# 3. ray assembly: d c2w / d c2w_staticcam / d rays_o, rays_d against float64 autograd of get_rays / ndc_rays / normalise / cat
# ---------------------------------------------------------------------------------------------------------------------------
def _dirs64(H, W, focal, window):
    """camera-frame directions of the window's pixels, float64 (run_nerf_helpers.get_rays casts the pose to fp32, so the
    reference is restated here in float64)"""
    i0, j0, h, w = window
    j, i = torch.meshgrid(torch.arange(i0, i0 + h, dtype=torch.float64), torch.arange(j0, j0 + w, dtype=torch.float64),
                          indexing="ij")
    return torch.stack([(i - W * .5) / focal, -(j - H * .5) / focal, -torch.ones_like(i)], -1).reshape(-1, 3)


def _rays64(dirs, pose):
    """pose [3,4] or one per pixel [n,3,4] -> rays_o, rays_d [n,3]"""
    R = pose[..., :3, :3]
    rays_d = (dirs[:, None, :] * R).sum(-1)
    return pose[..., :3, 3].expand(rays_d.shape), rays_d


def _assemble64(H, W, focal, near, far, ndc, use_vd, window, c2w=None, cs=None, rays=None):
    """the batch render() assembles (run.py:1171-1207), in float64; poses may be given per pixel ([n,3,4])"""
    from mvip_nerf_b200.run_nerf_helpers import ndc_rays
    if rays is None:
        dirs = _dirs64(H, W, focal, window)
        ro, rd = _rays64(dirs, c2w)
        vd = rd
        if cs is not None:
            ro, rd = _rays64(dirs, cs)
    else:
        ro, rd = rays
        vd = rd
    vd = vd / torch.norm(vd, dim=-1, keepdim=True)
    if ndc:
        ro, rd = ndc_rays(H, W, focal, 1., ro, rd)
    ones = torch.ones_like(rd[:, :1])
    return torch.cat([ro, rd, near * ones, far * ones] + ([vd] if use_vd else []), -1)


CASES = ["plain", "ndc", "ndc_static", "ndc_patch", "ndc_nodirs", "static", "patch"]
# Bar, relative to the sum over pixels of |per-pixel term| (for d rays_o / rays_d: to the ray's largest |term|): each term is an
# fp32 chain of at most ~40 roundings (get_rays, ndc_rays and the normalisation, forward and backward), i.e. <= 40 2^-24 of the
# magnitudes it combines; the NDC differences (d/d.z - o/o.z) can cancel, which we allow for with a factor 8; the pose sum adds at
# most (terms per thread + 5 warp levels + 8 warps + 592 blocks) 2^-24 of the absolute sum.  2^-13 covers both with margin.
ASM_REL = 2.0 ** -13


def _case(gd, c):
    H, W, focal, near, far, ndc, use_vd, i0, j0, h, w = gd[c + "_args"]
    return int(H), int(W), float(focal), float(near), float(far), bool(ndc), bool(use_vd), (int(i0), int(j0), int(h), int(w))


@pytest.mark.parametrize("case", CASES)
def test_ray_assembly_backward(case):
    import os
    from mvip_nerf_b200 import ops
    gd = np.load(os.path.join(os.path.dirname(__file__), "golden", "ray_batch.npz"))
    H, W, focal, near, far, ndc, use_vd, win = _case(gd, case)
    c2w = torch.from_numpy(gd[case + "_c2w"]).double()
    cs = torch.from_numpy(gd[case + "_c2w_static"]).double() if case + "_c2w_static" in gd else None
    stride = 11 if use_vd else 8
    n = win[2] * win[3]
    g = torch.Generator().manual_seed(CASES.index(case))
    g_out = torch.randn(n, stride, generator=g, dtype=torch.float64)
    # one pose copy per pixel: the gradient w.r.t. the copies is each pixel's term; their sum is d c2w
    cc = c2w.expand(n, 3, 4).clone().requires_grad_(True)
    ccs = None if cs is None else cs.expand(n, 3, 4).clone().requires_grad_(True)
    b64 = _assemble64(H, W, focal, near, far, ndc, use_vd, win, c2w=cc, cs=ccs)
    terms = torch.autograd.grad((b64 * g_out).sum(), [cc] + ([ccs] if ccs is not None else []))
    g_c, g_cs = ops.rays_from_pose_backward(c2w.float().to(DEV), None if cs is None else cs.float().to(DEV), H, W, focal, win,
                                            g_out.float().to(DEV), use_viewdirs=use_vd, ndc=ndc)
    for got, t in zip((g_c, g_cs), terms):
        err = (got.cpu().double() - t.sum(0)).abs()
        bar = ASM_REL * t.abs().sum(0)
        FRAC.append(("assembly_pose", case, float((err / bar.clamp_min(1e-300)).max())))
        assert (err <= bar).all(), float((err / bar.clamp_min(1e-300)).max())
    g_c2, _ = ops.rays_from_pose_backward(c2w.float().to(DEV), None if cs is None else cs.float().to(DEV), H, W, focal, win,
                                          g_out.float().to(DEV), use_viewdirs=use_vd, ndc=ndc)
    assert torch.equal(g_c, g_c2)
    # rays= form (no static camera there): per-ray d rays_o / d rays_d
    if case + "_rays_o" in gd:
        ro = torch.from_numpy(gd[case + "_rays_o"]).double().requires_grad_(True)
        rd = torch.from_numpy(gd[case + "_rays_d"]).double().requires_grad_(True)
        go = torch.randn(ro.shape[0], stride, generator=g, dtype=torch.float64)
        b64 = _assemble64(H, W, focal, near, far, ndc, use_vd, win, rays=(ro, rd))
        wo, wd = torch.autograd.grad((b64 * go).sum(), [ro, rd])
        k_o, k_d, _ = ops.rays_pack_backward(ro.detach().float().to(DEV), rd.detach().float().to(DEV), None, go.float().to(DEV),
                                             use_viewdirs=use_vd, ndc=ndc, H=H, W=W, focal=focal)
        for got, want in ((k_o, wo), (k_d, wd)):
            rel = (got.cpu().double() - want).abs().max(1)[0] / want.abs().max(1)[0].clamp_min(1e-300)
            FRAC.append(("assembly_rays", case, float(rel.max()) / ASM_REL))
            assert float(rel.max()) <= ASM_REL, float(rel.max())


# ---------------------------------------------------------------------------------------------------------------------------
# 4./5. end to end through render(): against float64 autograd of the reference port, and nothing else moves
# ---------------------------------------------------------------------------------------------------------------------------
def _kwargs(nc, nf):
    from mvip_nerf_b200.run import _FusedQuery
    from mvip_nerf_b200.run_nerf_helpers import get_embedder
    e, _ = get_embedder(10)
    ev, _ = get_embedder(4)
    return dict(network_query_fn=_FusedQuery(e, ev, 65536), network_fn=nc, network_fine=nf, N_samples=64, N_importance=64,
                perturb=0., raw_noise_std=0., white_bkgd=True, lindisp=True, use_viewdirs=True, ndc=False)


def _trained():
    import os
    d = np.load(os.path.join(os.path.dirname(__file__), "golden", "trained_ckpt.npz"))
    nets = []
    for pre in ("coarse.", "fine."):
        net = _net(0)
        with torch.no_grad():
            for k, p in net.named_parameters():
                p.copy_(torch.from_numpy(d[pre + k]))
        net.invalidate_packed()
        nets.append(net)
    return d, nets


def _render_pose(kw, H, W, focal, near, far, c2w, patch, chunk=1 << 15):
    from mvip_nerf_b200.run import render
    rgb, disp, acc, depth, ex = render(H, W, focal, chunk=chunk, c2w=c2w, near=near, far=far, patch=patch, **kw)
    return rgb, ex


def _cos_rel(got, want):
    got, want = got.reshape(-1), want.reshape(-1)
    return float((got * want).sum() / (got.norm() * want.norm())), float((got - want).norm() / want.norm())


# bars: about 1.5x the deviation measured on a B200 (1000 W), as (min cos, max rel-L2) per (network, entry, gradient)
E2E_BARS = {("random", "c2w", "c2w"): (0.996, 0.11), ("trained", "c2w", "c2w"): (0.987, 0.20),
            ("random", "rays", "rays_o"): (0.9954, 0.118), ("random", "rays", "rays_d"): (0.9954, 0.118),
            ("trained", "rays", "rays_o"): (0.948, 0.40), ("trained", "rays", "rays_d"): (0.948, 0.40)}


@pytest.mark.parametrize("entry", ["c2w", "rays"])
@pytest.mark.parametrize("which", ["random", "trained"])
def test_render_grad_vs_reference(which, entry):
    from mvip_nerf_b200.run import render
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
    patch = (H // 4, W // 4, 16, 16)
    kw = _kwargs(nc, nf)
    g = torch.Generator().manual_seed(3)
    g_rgb = torch.randn(256, 3, generator=g, dtype=torch.float64)
    # float64 reference: the port's render_rays on the float64 ray batch (same depths: perturb 0, deterministic fine samples)
    if entry == "c2w":
        leaves = [c2w0.clone().requires_grad_(True)]
        b64 = _assemble64(H, W, focal, near, far, False, True, patch, c2w=leaves[0])
    else:
        ro64, rd64 = _rays64(_dirs64(H, W, focal, patch), c2w0)
        leaves = [ro64.detach().clone().requires_grad_(True), rd64.detach().clone().requires_grad_(True)]
        b64 = _assemble64(H, W, focal, near, far, False, True, patch, rays=tuple(leaves))
    pc = {k: v.double() for k, v in port.params_from_numpy(_params_np(nc)).items()}
    pf = {k: v.double() for k, v in port.params_from_numpy(_params_np(nf)).items()}
    out = port.render_rays(b64, pc, pf, torch.linspace(0., 1., 64, dtype=torch.float64), lindisp=True, white_bkgd=True)
    # rays whose reference density at the last sample is within 5e-3 of zero are ill-conditioned (dist 1e10): no upstream gradient
    with torch.no_grad():
        pts = b64[:, None, 0:3] + b64[:, None, 3:6] * out["z_vals"][..., None]
        keep = (port.query(pf, pts, b64[:, -3:])[:, -1, 3].abs() > 5e-3).double()[:, None]
    wants = torch.autograd.grad((out["rgb_map"] * g_rgb * keep).sum(), leaves)
    # the kernels, through render()
    if entry == "c2w":
        ins = [c2w0.float().to(DEV).requires_grad_(True)]
        rgb, _, _, _, _ = render(H, W, focal, c2w=ins[0], near=near, far=far, patch=patch, **kw)
    else:
        ins = [leaves[0].detach().float().to(DEV).requires_grad_(True), leaves[1].detach().float().to(DEV).requires_grad_(True)]
        rgb, _, _, _, _ = render(H, W, focal, rays=tuple(ins), near=near, far=far, **kw)
    (rgb.reshape(-1, 3).double() * (g_rgb * keep).to(DEV)).sum().backward()
    names = ["c2w"] if entry == "c2w" else ["rays_o", "rays_d"]
    res = []
    for name, x, want in zip(names, ins, wants):
        got = x.grad.double().cpu()
        assert torch.isfinite(got).all()
        cos, rel = _cos_rel(got, want)
        FRAC.append(("e2e", which, entry, name, int(keep.sum()), cos, rel))
        res.append((name, cos, rel))
    for name, cos, rel in res:
        min_cos, max_rel = E2E_BARS[(which, entry, name)]
        assert cos > min_cos and rel < max_rel, (name, cos, rel)


# entries that only the gradient w.r.t. rays / poses calls, and their launches per call in render()'s rays mode; the compositing
# backward with d rays_d takes the place of the plain one (one launch either way)
NEW_ENTRIES = {"mvip_mlp_input_grad": 2, "mvip_rays_from_pose_backward": 2, "mvip_rays_pack_backward": 1}
REPLACING = {"mvip_composite_backward_rays": "mvip_composite_backward"}


def test_nothing_else_moves():
    from mvip_nerf_b200 import ops
    from mvip_nerf_b200.run import render, render_deferred
    nc, nf = _net(21), _net(22)
    kw = _kwargs(nc, nf)
    H, W, focal = 48, 64, 60.0
    c2w0 = torch.tensor([[1, 0, 0, 0.1], [0, 1, 0, -0.2], [0, 0, 1, 4.0]], device=DEV)

    def run(pose_grad, deferred=False, chunk=1024):
        for net in (nc, nf):
            for p in net.parameters():
                p.grad = None
        fwd, bwd = [], []
        calls = fwd
        real = ops._call

        def spy(name, *a):
            calls.append(name if isinstance(name, str) else name[0])
            return real(name, *a)
        n0 = ops.launch_count
        ops._call = spy
        try:
            c = c2w0.clone().requires_grad_(pose_grad)
            fn = render_deferred if deferred else render
            rgb, disp, acc, depth, ex = fn(H, W, focal, chunk=chunk, c2w=c, near=2., far=6., **kw)
            g = torch.linspace(-1, 1, rgb.numel(), device=DEV).view(rgb.shape)
            calls = bwd
            ((rgb * g).sum() + (ex["rgb0"] * g).sum()).backward()   # rgb0: the coarse network gets nothing through the fine depths
        finally:
            ops._call = real
        grads = [p.grad.clone() for net in (nc, nf) for p in net.parameters()]
        return rgb.detach(), grads, (c.grad.clone() if pose_grad else None), (fwd, bwd), ops.launch_count - n0

    from collections import Counter
    run(False)    # packs the bf16 weights (the first forward of a network does), so that both runs below find them packed
    rgb0, g0, _, (f0, b0), n0 = run(False)
    # no input requires grad: none of the new entries runs, so the launches are those of the code without them
    assert not any(n in NEW_ENTRIES or n in REPLACING for n in f0 + b0)
    rgb1, g1, dc1, (f1, b1), n1 = run(True)
    # with a pose gradient: the forward issues the same entries in the same order; the backward issues the same entries (the
    # compositing backward in its d rays_d form) plus the new ones (autograd orders independent nodes itself, and the ray batch
    # joining the graph changes that order); the launch count grows by exactly the new entries' launches
    assert f1 == f0
    assert Counter(REPLACING.get(n, n) for n in b1 if n not in NEW_ENTRIES) == Counter(b0)
    assert n1 - n0 == sum(NEW_ENTRIES[n] for n in b1 if n in NEW_ENTRIES)
    assert torch.equal(rgb0, rgb1), "rendered maps moved"
    assert all(torch.equal(a, b) for a, b in zip(g0, g1)), "parameter gradients moved"
    _, _, dc2, _, _ = run(True)
    assert torch.equal(dc1, dc2), "d c2w not reproducible"
    assert torch.isfinite(dc1).all() and dc1.abs().sum() > 0
    _, _, dcd, _, _ = run(True, deferred=True)
    assert torch.equal(dcd, dc1), (dcd, dc1)


def test_nerf_forward_on_embedded_inputs_gives_no_input_gradient():
    """NeRF.forward(x) re-encodes columns 0:3 / 63:66 of x on chip, so it cannot give the reference's gradient for x: x gets
    none (as before), the parameter gradients are those of a detached x, and no input-gradient kernel runs."""
    from mvip_nerf_b200 import ops
    from mvip_nerf_b200.run_nerf_helpers import get_embedder
    net = _net(31)
    e, _ = get_embedder(10)
    ev, _ = get_embedder(4)
    g = torch.Generator(device=DEV).manual_seed(5)
    pts = torch.randn(1000, 3, device=DEV, generator=g)
    dirs = torch.nn.functional.normalize(torch.randn(1000, 3, device=DEV, generator=g), dim=-1)
    x0 = torch.cat([e(pts), ev(dirs)], -1)
    up = torch.randn(1000, 4, device=DEV, generator=g)

    def run(x):
        for p in net.parameters():
            p.grad = None
        (net(x) * up).sum().backward()
        return [p.grad.clone() for p in net.parameters()]
    ref = run(x0.clone())
    calls = []
    real = ops._call
    ops._call = lambda name, *a: (calls.append(name), real(name, *a))[1]
    try:
        x = x0.clone().requires_grad_(True)
        got = run(x)
    finally:
        ops._call = real
    assert x.grad is None
    assert "mvip_mlp_input_grad" not in calls
    assert all(torch.equal(a, b) for a, b in zip(ref, got))


# ---------------------------------------------------------------------------------------------------------------------------
# 6. camera refinement against a frozen trained network (iNeRF-style)
# ---------------------------------------------------------------------------------------------------------------------------
def _rodrigues(w):
    th = w.norm()
    k = w / th
    K = torch.tensor([[0, -k[2], k[1]], [k[2], 0, -k[0]], [-k[1], k[0], 0]], dtype=w.dtype, device=w.device)
    return torch.eye(3, dtype=w.dtype, device=w.device) + torch.sin(th) * K + (1 - torch.cos(th)) * K @ K


STEPS = 200


def test_pose_refinement_converges():
    """Adam on a pose correction (axis-angle + translation) through render(c2w=...), target = the frozen trained networks'
    rendering at the golden pose, four 48 x 48 patches (one per image quadrant) per step; start 1 degree and 1 % of the depth
    range off."""
    d, (nc, nf) = _trained()
    for net in (nc, nf):
        for p in net.parameters():
            p.requires_grad_(False)
    H, W, focal, near, far = int(d["H"]), int(d["W"]), float(d["focal"]), float(d["near"]), float(d["far"])
    kw = _kwargs(nc, nf)
    c2w_true = torch.from_numpy(d["c2w"]).float().to(DEV)
    patches = [(H // 4 - 24 + (H // 2) * a, W // 4 - 24 + (W // 2) * b, 48, 48) for a in (0, 1) for b in (0, 1)]

    def render_all(c):
        return torch.cat([_render_pose(kw, H, W, focal, near, far, c, pt)[0].reshape(-1, 3) for pt in patches], 0)
    with torch.no_grad():
        target = render_all(c2w_true)
    R_err = _rodrigues(torch.tensor([0.0, 1.0, 0.5], device=DEV) / 1.118 * np.deg2rad(1.0))
    dt = torch.tensor([1.0, -1.0, 0.5], device=DEV) / 1.5 * 0.01 * (far - near)
    rot = torch.nn.Parameter(torch.zeros(3, device=DEV))
    trans = torch.nn.Parameter(torch.zeros(3, device=DEV))
    opt = torch.optim.Adam([rot, trans], lr=2e-3)
    sched = torch.optim.lr_scheduler.CosineAnnealingLR(opt, STEPS)
    base = torch.cat([R_err @ c2w_true[:, :3], (c2w_true[:, 3] + dt)[:, None]], 1)

    def pose():
        th = rot.norm() + 1e-12
        k = rot / th
        zero = torch.zeros((), device=DEV)
        K = torch.stack([torch.stack([zero, -k[2], k[1]]), torch.stack([k[2], zero, -k[0]]), torch.stack([-k[1], k[0], zero])])
        Rr = torch.eye(3, device=DEV) + torch.sin(th) * K + (1 - torch.cos(th)) * K @ K
        return torch.cat([Rr @ base[:, :3], (base[:, 3] + trans)[:, None]], 1)

    def errs(c):
        Rrel = c[:, :3].detach() @ c2w_true[:, :3].T
        ang = float(torch.arccos(((torch.trace(Rrel) - 1) / 2).clamp(-1, 1)))
        return ang, float((c[:, 3].detach() - c2w_true[:, 3]).norm())

    a0, t0 = errs(pose())
    losses = []
    for _ in range(STEPS):
        opt.zero_grad()
        loss = ((render_all(pose()) - target) ** 2).mean()
        loss.backward()
        opt.step()
        sched.step()
        losses.append(float(loss.detach()))
    a1, t1 = errs(pose())
    FRAC.append(("refine", STEPS, a1 / a0, t1 / t0, losses[0], losses[-1]))
    assert losses[-1] < 0.5 * losses[0]
    assert a1 <= 0.5 * a0 and t1 <= 0.5 * t0, (a0, a1, t0, t1)


def test_record_fractions():
    """writes the measured fractions of the bars (and the end-to-end figures) when MVIP_POSE_GRAD_OUT is set"""
    import json
    import os
    out = os.environ.get("MVIP_POSE_GRAD_OUT")
    if out:
        with open(out, "w") as f:
            json.dump([list(r) for r in FRAC], f, indent=1)
