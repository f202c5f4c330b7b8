"""Thin torch-tensor wrappers over the C ABI (include/mvip_nerf.h).

PyTorch is plumbing only: it owns device memory and the stream; every computation below is one of
our sm_100a kernels in libmvip_nerf.so.  Inputs must be CUDA tensors — there is no CPU path.
"""
import ctypes
import os

import torch

from . import _lib

PARAM_ORDER = (["pts_linears.%d.%s" % (i, k) for i in range(8) for k in ("weight", "bias")] +
               ["views_linears.0.weight", "views_linears.0.bias", "feature_linear.weight", "feature_linear.bias",
                "alpha_linear.weight", "alpha_linear.bias", "rgb_linear.weight", "rgb_linear.bias"])
PARAM_SHAPES = ([(256, 63), (256,)] + [(256, 256), (256,)] * 4 + [(256, 319), (256,)] + [(256, 256), (256,)] * 2 +
                [(128, 283), (128,), (256, 256), (256,), (1, 256), (1,), (3, 128), (3,)])

# kernel launches issued through this module (bench.py reports it as gpu_launches)
launch_count = 0
# bumped by optim.FusedAdam.step(): parameters changed in place without torch's version counters noticing
param_epoch = 0
_LAUNCHES = {"mvip_rays_from_pose": 1, "mvip_rays_from_pose_ndc": 1, "mvip_rays_pack": 1, "mvip_sample_coarse": 1, "mvip_sample_pdf": 1, "mvip_sample_fine": 1, "mvip_composite_forward": 1,
             "mvip_composite_backward": 1, "mvip_composite_forward_mse": 1, "mvip_composite_backward_mse": 1, "mvip_normal_forward": 2, "mvip_normal_backward": 4, "mvip_normal_forward_xyz": 2, "mvip_normal_backward_xyz": 4, "mvip_embed": 1,
             "mvip_mlp_pack_weights": 1, "mvip_mlp_forward": 1, "mvip_mlp_backward": 3, "mvip_selftest_umma": 1,
             "mvip_rays_pack_backward": 1, "mvip_rays_from_pose_backward": 2, "mvip_composite_backward_rays": 1,
             "mvip_mlp_input_grad": 1, "mvip_rays_from_poses": 1, "mvip_rays_from_poses_backward": 2}


class _KernelTimer:
    """Optional CUDA-event bracket around every library call (bench.py: per-kernel times inside the timed region)."""

    def __init__(self):
        self.on = False
        self.recs = []

    def enable(self, on):
        self.on = bool(on)
        if on:
            self.recs = []

    def collect(self):
        torch.cuda.synchronize()
        out = {}
        for name, e0, e1 in self.recs:
            out.setdefault(name, []).append(e0.elapsed_time(e1))
        self.recs = []
        return out


kernel_timer = _KernelTimer()


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _f32(t, name):
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError("%s must be a CUDA tensor: mvip_nerf_b200 has no CPU fallback" % name)
    if t.dtype != torch.float32:
        t = t.float()
    return t.contiguous()


def _rows3(t, name):
    """[N, >=3] fp32 CUDA rows read through a row stride (e.g. the rays_d columns of the ray batch): no copy."""
    if t.is_cuda and t.dtype == torch.float32 and t.dim() == 2 and t.stride(1) == 1 and t.shape[0] > 0:
        return t, t.stride(0)
    t = _f32(t, name)
    return t, t.shape[-1]


def _call(name, *args):
    global launch_count
    lib = _lib.load()
    label = None
    if isinstance(name, tuple):
        name, label = name
    if kernel_timer.on:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        rc = getattr(lib, name)(*args)
        e1.record()
        kernel_timer.recs.append((label or name, e0, e1))
    else:
        rc = getattr(lib, name)(*args)
    _lib.check(rc, name)
    launch_count += 1 if label else _LAUNCHES.get(name, 1)


# ---------------------------------------------------------------------------------------------- rays
def rays_from_pose(H, W, focal, c2w, near, far, use_viewdirs=True, c2w_staticcam=None, patch=None, device=None, ndc=False,
                   ndc_near=1.):
    """-> ray batch [h*w, 8 | 11] (o, d, near, far[, viewdir]) of a pinhole view   (get_rays [+ ndc_rays] + run.py:1171-1207)"""
    def pose(x):
        if x is None:
            return None
        t = torch.as_tensor(x, dtype=torch.float32)
        dev = device or (t.device if t.is_cuda else torch.device("cuda", torch.cuda.current_device()))
        return t.to(dev)[:3, :4].contiguous()
    c = pose(c2w)
    cs = pose(c2w_staticcam)
    i0, j0, h, w = (0, 0, H, W) if patch is None else [int(v) for v in patch]
    out = torch.empty((h * w, 11 if use_viewdirs else 8), device=c.device, dtype=torch.float32)
    _call("mvip_rays_from_pose_ndc", _ptr(c), _ptr(cs), int(H), int(W), float(focal), float(near), float(far), i0, j0, h, w,
          int(bool(use_viewdirs)), int(bool(ndc)), float(ndc_near), _ptr(out), _stream())
    return out


def rays_pack(rays_o, rays_d, near, far, use_viewdirs=True, view_d=None, ndc=False, H=0, W=0, focal=1., ndc_near=1.):
    """rays_o / rays_d [n,3] -> ray batch [n, 8 | 11]   (the `rays=` entry of render(), run.py:1176-1207)"""
    rays_o = _f32(rays_o, "rays_o").reshape(-1, 3)
    rays_d = _f32(rays_d, "rays_d").reshape(-1, 3)
    view_d = None if view_d is None else _f32(view_d, "view_d").reshape(-1, 3)
    n = rays_d.shape[0]
    if rays_o.shape[0] != n or (view_d is not None and view_d.shape[0] != n):
        raise RuntimeError("rays_o / rays_d / view_d row counts differ")
    out = torch.empty((n, 11 if use_viewdirs else 8), device=rays_d.device, dtype=torch.float32)
    _call("mvip_rays_pack", _ptr(rays_o), _ptr(rays_d), _ptr(view_d), n, float(near), float(far), int(bool(use_viewdirs)),
          int(bool(ndc)), int(H), int(W), float(focal), float(ndc_near), _ptr(out), _stream())
    return out


def rays_pack_backward(rays_o, rays_d, view_d, g_out, use_viewdirs=True, ndc=False, H=0, W=0, focal=1., ndc_near=1.):
    """gradient of rays_pack: g_out [n, 8 | 11] -> (d rays_o, d rays_d, d view_d | None), each [n,3]"""
    rays_o = _f32(rays_o, "rays_o").reshape(-1, 3)
    rays_d = _f32(rays_d, "rays_d").reshape(-1, 3)
    view_d = None if view_d is None else _f32(view_d, "view_d").reshape(-1, 3)
    g_out = _f32(g_out, "g_out")
    n = rays_d.shape[0]
    g_o, g_d = torch.empty_like(rays_o), torch.empty_like(rays_d)
    g_v = None if view_d is None else torch.empty_like(view_d)
    _call("mvip_rays_pack_backward", _ptr(rays_o), _ptr(rays_d), _ptr(view_d), n, int(bool(use_viewdirs)), int(bool(ndc)), int(H),
          int(W), float(focal), float(ndc_near), _ptr(g_out), _ptr(g_o), _ptr(g_d), _ptr(g_v), _stream())
    return g_o, g_d, g_v


def rays_from_pose_backward(c2w, c2w_staticcam, H, W, focal, window, g_out, use_viewdirs=True, ndc=False, ndc_near=1.):
    """gradient of rays_from_pose: g_out [h*w, 8 | 11] -> (d c2w [3,4], d c2w_staticcam [3,4] | None); window = (i0, j0, h, w)"""
    c2w = _f32(c2w, "c2w")
    cs = _f32(c2w_staticcam, "c2w_staticcam")
    g_out = _f32(g_out, "g_out")
    i0, j0, h, w = [int(v) for v in window]
    g_c = torch.empty((3, 4), device=c2w.device, dtype=torch.float32)
    g_cs = None if cs is None else torch.empty((3, 4), device=c2w.device, dtype=torch.float32)
    ws = torch.empty((_lib.load().mvip_rays_from_pose_backward_workspace_bytes() // 4,), device=c2w.device, dtype=torch.float32)
    _call("mvip_rays_from_pose_backward", _ptr(c2w), _ptr(cs), int(H), int(W), float(focal), i0, j0, h, w, int(bool(use_viewdirs)),
          int(bool(ndc)), float(ndc_near), _ptr(g_out), _ptr(g_c), _ptr(g_cs), _ptr(ws), _stream())
    return g_c, g_cs


def _poses_arg(poses):
    """[V,3,4] or [V,4,4] fp32 CUDA pose table -> contiguous [V,3,4]"""
    p = _f32(poses, "poses")
    if p.dim() != 3 or p.shape[1] not in (3, 4) or p.shape[2] != 4:
        raise RuntimeError("poses must be [V,3,4] or [V,4,4], got %s" % (tuple(p.shape),))
    return p[:, :3, :].contiguous()


def _pixels_arg(pixels):
    """[N,3] (view, row, col) CUDA indices, int32 or int64 -> contiguous int32 (int64 values outside int32 stay out of range)"""
    if not pixels.is_cuda:
        raise RuntimeError("pixels must be a CUDA tensor: mvip_nerf_b200 has no CPU fallback")
    if pixels.dim() != 2 or pixels.shape[1] != 3:
        raise RuntimeError("pixels must be [N,3] = (view, row, col), got %s" % (tuple(pixels.shape),))
    if pixels.dtype == torch.int64:
        pixels = pixels.clamp(-1, 2 ** 31 - 1).to(torch.int32)
    elif pixels.dtype != torch.int32:
        raise RuntimeError("pixels must be int32 or int64, got %s" % pixels.dtype)
    return pixels.contiguous()


def rays_from_poses(H, W, focal, poses, pixels, near, far, use_viewdirs=True, ndc=False, ndc_near=1.):
    """pose table [V,3,4] + pixels [N,3] = (view, row, col) -> ray batch [N, 8 | 11]; row k equals row row*W + col of
    rays_from_pose(poses[view]) over the whole image, bitwise.  Out-of-range entries give rows of NaN."""
    poses = _poses_arg(poses)
    pixels = _pixels_arg(pixels)
    n = pixels.shape[0]
    out = torch.empty((n, 11 if use_viewdirs else 8), device=pixels.device, dtype=torch.float32)
    _call("mvip_rays_from_poses", _ptr(poses), poses.shape[0], _ptr(pixels), n, int(H), int(W), float(focal), float(near), float(far),
          int(bool(use_viewdirs)), int(bool(ndc)), float(ndc_near), _ptr(out), _stream())
    return out


def rays_from_poses_backward(poses, pixels, H, W, focal, g_out, use_viewdirs=True, ndc=False, ndc_near=1.):
    """gradient of rays_from_poses: g_out [N, 8 | 11] -> d poses [V,3,4] (views no entry uses get 0)"""
    poses = _poses_arg(poses)
    pixels = _pixels_arg(pixels)
    g_out = _f32(g_out, "g_out")
    V, n = poses.shape[0], pixels.shape[0]
    g_p = torch.empty((V, 3, 4), device=poses.device, dtype=torch.float32)
    ws = torch.empty((max(1, _lib.load().mvip_rays_from_poses_backward_workspace_bytes(n, V) // 4),), device=poses.device,
                     dtype=torch.float32)
    _call("mvip_rays_from_poses_backward", _ptr(poses), V, _ptr(pixels), n, int(H), int(W), float(focal), int(bool(use_viewdirs)),
          int(bool(ndc)), float(ndc_near), _ptr(g_out), _ptr(g_p), _ptr(ws), _stream())
    return g_p


# ---------------------------------------------------------------------------------------------- sampling
def sample_coarse(rays, t_vals, t_rand=None, lindisp=False):
    """rays [N,>=8] -> z_vals [N,S]   (run.py:1759-1781)"""
    rays = _f32(rays, "rays")
    t_vals = _f32(t_vals, "t_vals")
    t_rand = _f32(t_rand, "t_rand")
    N, S = rays.shape[0], t_vals.numel()
    z = torch.empty((N, S), device=rays.device, dtype=torch.float32)
    _call("mvip_sample_coarse", _ptr(rays), rays.shape[1], N, _ptr(t_vals), _ptr(t_rand), S, int(bool(lindisp)),
          _ptr(z), _stream())
    return z


def _u_arg(u, n_rows):
    u = _f32(u, "u")
    if u.dim() == 1:
        return u, 1, u.numel()
    if u.shape[0] != n_rows:
        raise RuntimeError("u has %d rows, expected %d" % (u.shape[0], n_rows))
    return u, 0, u.shape[-1]


def sample_pdf(bins, weights, u, want_inds=False, want_cdf=False):
    """(run_nerf_helpers.py:304-347) bins [N,B], weights [N,B-1], u [N,M] or [M] -> samples [N,M] (+inds, +cdf)"""
    bins = _f32(bins, "bins")
    weights = _f32(weights, "weights")
    N, B = bins.shape
    if weights.shape != (N, B - 1):
        raise RuntimeError("weights must be [N, n_bins-1]")
    u, is_row, M = _u_arg(u, N)
    samples = torch.empty((N, M), device=bins.device, dtype=torch.float32)
    inds = torch.empty((N, M), device=bins.device, dtype=torch.int64) if want_inds else None
    cdf = torch.empty((N, B), device=bins.device, dtype=torch.float32) if want_cdf else None
    _call("mvip_sample_pdf", _ptr(bins), _ptr(weights), _ptr(u), is_row, N, B, M, _ptr(samples), _ptr(inds), _ptr(cdf),
          _stream())
    return samples, inds, cdf


def sample_fine(z_vals, weights, u, want_samples=True, want_inds=False, want_std=True):
    """(run.py:1809-1816,1836) -> dict(z_samples, inds, z_merged, z_std)"""
    z_vals = _f32(z_vals, "z_vals")
    weights = _f32(weights, "weights")
    N, S = z_vals.shape
    u, is_row, M = _u_arg(u, N)
    dev = z_vals.device
    z_samples = torch.empty((N, M), device=dev, dtype=torch.float32) if want_samples else None
    inds = torch.empty((N, M), device=dev, dtype=torch.int64) if want_inds else None
    z_std = torch.empty((N,), device=dev, dtype=torch.float32) if want_std else None
    z_merged = torch.empty((N, S + M), device=dev, dtype=torch.float32)
    _call("mvip_sample_fine", _ptr(z_vals), _ptr(weights), _ptr(u), is_row, N, S, M, _ptr(z_samples), _ptr(inds),
          _ptr(z_merged), _ptr(z_std), _stream())
    return {"z_samples": z_samples, "inds": inds, "z_merged": z_merged, "z_std": z_std}


# ---------------------------------------------------------------------------------------------- compositing
_mse_ws = {}


def _mse_workspace(dev):
    """ticket counter + per-block partials of the fused-loss forward: zero-filled once per device, reused by every call"""
    ws = _mse_ws.get(dev)
    if ws is None:
        ws = _mse_ws[dev] = torch.zeros(_lib.load().mvip_composite_mse_workspace_bytes() // 4, device=dev, dtype=torch.float32)
    return ws


def composite_forward(raw, z_vals, rays_d, noise=None, white_bkgd=False, need_alpha=False, target_rgb=None, target_disp=None):
    """-> (rgb, disp, acc, weights, depth, alpha | None) [+ sq [2] = (sum (rgb - target_rgb)^2, sum (disp - target_disp)^2) when a
    target is given: img2mse fused into the kernel, DS_NeRF/run.py:1000-1027]"""
    raw = _f32(raw, "raw")
    z_vals = _f32(z_vals, "z_vals")
    rays_d, d_stride = _rows3(rays_d, "rays_d")
    noise = _f32(noise, "noise")
    N, S = z_vals.shape
    dev = raw.device
    rgb = torch.empty((N, 3), device=dev, dtype=torch.float32)
    disp = torch.empty((N,), device=dev, dtype=torch.float32)
    acc = torch.empty((N,), device=dev, dtype=torch.float32)
    depth = torch.empty((N,), device=dev, dtype=torch.float32)
    weights = torch.empty((N, S), device=dev, dtype=torch.float32)
    alpha = torch.empty((N, S), device=dev, dtype=torch.float32) if need_alpha else None
    if target_rgb is not None or target_disp is not None:
        target_rgb, target_disp = _f32(target_rgb, "target_rgb"), _f32(target_disp, "target_disp")
        if (target_rgb is not None and target_rgb.numel() != 3 * N) or (target_disp is not None and target_disp.numel() != N):
            raise RuntimeError("fused-loss targets must have one row per ray")
        sq = torch.empty((2,), device=dev, dtype=torch.float32)
        _call("mvip_composite_forward_mse", _ptr(raw), _ptr(z_vals), _ptr(rays_d), d_stride, _ptr(noise), N, S, int(bool(white_bkgd)),
              _ptr(target_rgb), _ptr(target_disp), _ptr(rgb), _ptr(disp), _ptr(acc), _ptr(weights), _ptr(depth), _ptr(alpha), _ptr(sq),
              _ptr(_mse_workspace(dev)), _stream())
        return rgb, disp, acc, weights, depth, alpha, sq
    _call("mvip_composite_forward", _ptr(raw), _ptr(z_vals), _ptr(rays_d), d_stride, _ptr(noise), N, S,
          int(bool(white_bkgd)), _ptr(rgb), _ptr(disp), _ptr(acc), _ptr(weights), _ptr(depth), _ptr(alpha), _stream())
    return rgb, disp, acc, weights, depth, alpha


def composite_backward(raw, z_vals, rays_d, noise, white_bkgd, detach_weights, g_rgb, g_disp, g_acc, g_depth,
                       g_weights=None, g_alpha=None, target_rgb=None, target_disp=None, g_sq=None, want_rays_d=False):
    """-> d_raw [N,S,4]; with want_rays_d -> (d_raw, d rays_d [N,3])"""
    raw = _f32(raw, "raw")
    z_vals = _f32(z_vals, "z_vals")
    rays_d, d_stride = _rows3(rays_d, "rays_d")
    N, S = z_vals.shape
    d_raw = torch.empty((N, S, 4), device=raw.device, dtype=torch.float32)
    args = [_f32(t, "grad") for t in (g_rgb, g_disp, g_acc, g_depth, g_weights, g_alpha)]
    if want_rays_d:
        fused = g_sq is not None and (target_rgb is not None or target_disp is not None)
        d_dir = torch.empty((N, 3), device=raw.device, dtype=torch.float32)
        _call("mvip_composite_backward_rays", _ptr(raw), _ptr(z_vals), _ptr(rays_d), d_stride, _ptr(_f32(noise, "noise")), N, S,
              int(bool(white_bkgd)), int(bool(detach_weights)), _ptr(_f32(target_rgb, "target_rgb") if fused else None),
              _ptr(_f32(target_disp, "target_disp") if fused else None), _ptr(_f32(g_sq, "g_sq") if fused else None),
              *[_ptr(a) for a in args], _ptr(d_raw), _ptr(d_dir), _stream())
        return d_raw, d_dir
    if g_sq is not None and (target_rgb is not None or target_disp is not None):
        _call("mvip_composite_backward_mse", _ptr(raw), _ptr(z_vals), _ptr(rays_d), d_stride, _ptr(_f32(noise, "noise")), N, S,
              int(bool(white_bkgd)), int(bool(detach_weights)), _ptr(_f32(target_rgb, "target_rgb")), _ptr(_f32(target_disp, "target_disp")),
              _ptr(_f32(g_sq, "g_sq")), *[_ptr(a) for a in args], _ptr(d_raw), _stream())
        return d_raw
    _call("mvip_composite_backward", _ptr(raw), _ptr(z_vals), _ptr(rays_d), d_stride, _ptr(_f32(noise, "noise")),
          N, S, int(bool(white_bkgd)), int(bool(detach_weights)), *[_ptr(a) for a in args], _ptr(d_raw), _stream())
    return d_raw


# ---------------------------------------------------------------------------------------------- normal map
def _normal_ws(H, W, dev):
    n = _lib.load().mvip_normal_workspace_bytes(H, W)
    return torch.empty((n // 8,), device=dev, dtype=torch.float64)


def normal_forward(depth, fx, fy, cx, cy, k=31):
    depth = _f32(depth, "depth")
    H, W = depth.shape
    normal = torch.empty((3, H, W), device=depth.device, dtype=torch.float32)
    ws = _normal_ws(H, W, depth.device)
    _call("mvip_normal_forward", _ptr(depth), H, W, float(fx), float(fy), float(cx), float(cy), int(k), _ptr(normal),
          _ptr(ws), _stream())
    return normal


def normal_backward(depth, fx, fy, cx, cy, g_normal, k=31):
    depth = _f32(depth, "depth")
    g_normal = _f32(g_normal, "g_normal")
    H, W = depth.shape
    d_depth = torch.empty((H, W), device=depth.device, dtype=torch.float32)
    ws = _normal_ws(H, W, depth.device)
    _call("mvip_normal_backward", _ptr(depth), H, W, float(fx), float(fy), float(cx), float(cy), int(k), _ptr(g_normal),
          _ptr(d_depth), _ptr(ws), _stream())
    return d_depth


def normal_forward_xyz(xyz, k=31):
    """xyz [3,H,W] -> normal [3,H,W]   (depth2normal_geo, run.py:1924-1940)"""
    xyz = _f32(xyz, "xyz")
    _, H, W = xyz.shape
    normal = torch.empty((3, H, W), device=xyz.device, dtype=torch.float32)
    ws = _normal_ws(H, W, xyz.device)
    _call("mvip_normal_forward_xyz", _ptr(xyz), H, W, int(k), _ptr(normal), _ptr(ws), _stream())
    return normal


def normal_backward_xyz(xyz, g_normal, k=31):
    xyz = _f32(xyz, "xyz")
    g_normal = _f32(g_normal, "g_normal")
    _, H, W = xyz.shape
    d_xyz = torch.empty((3, H, W), device=xyz.device, dtype=torch.float32)
    ws = _normal_ws(H, W, xyz.device)
    _call("mvip_normal_backward_xyz", _ptr(xyz), H, W, int(k), _ptr(g_normal), _ptr(d_xyz), _ptr(ws), _stream())
    return d_xyz


# ---------------------------------------------------------------------------------------------- embedding
def embed(x, num_freqs):
    """x [..., D] -> [..., D*(1+2L)]   (Embedder.embed, run_nerf_helpers.py:51-52)"""
    if not x.is_cuda:
        raise RuntimeError("x must be a CUDA tensor: mvip_nerf_b200 has no CPU fallback")
    D = x.shape[-1]
    flat = x.reshape(-1, D)
    if flat.dtype != torch.float32:
        flat = flat.float()
    if flat.stride(-1) != 1:
        flat = flat.contiguous()
    n = flat.shape[0]
    out = torch.empty((n, D * (1 + 2 * num_freqs)), device=x.device, dtype=torch.float32)
    _call("mvip_embed", _ptr(flat), flat.stride(0) if n > 0 else D, n, D, int(num_freqs), _ptr(out), _stream())
    return out.reshape(*x.shape[:-1], out.shape[-1])


# ---------------------------------------------------------------------------------------------- MLP
def _aligned_bytes(nbytes, dev):
    """uint8 buffer whose data_ptr is 1024-byte aligned (torch's caching allocator gives >= 512)."""
    buf = torch.empty((nbytes + 1024,), device=dev, dtype=torch.uint8)
    off = (-buf.data_ptr()) % 1024
    return buf[off:off + nbytes]


def mlp_pack(params, out=None):
    """params: sequence of 24 fp32 CUDA tensors in PARAM_ORDER -> packed uint8 blob"""
    lib = _lib.load()
    ps = [_f32(p.detach(), "param") for p in params]
    if len(ps) != _lib.MVIP_MLP_NUM_PARAMS:
        raise RuntimeError("expected %d parameter tensors" % _lib.MVIP_MLP_NUM_PARAMS)
    for t, shp, name in zip(ps, PARAM_SHAPES, PARAM_ORDER):
        if tuple(t.shape) != shp:
            raise RuntimeError("%s has shape %s, the fused kernels need %s (D=8, W=256, multires=10/4, skips=[4], "
                               "use_viewdirs)" % (name, tuple(t.shape), shp))
    if out is None:
        out = _aligned_bytes(lib.mvip_mlp_packed_bytes(), ps[0].device)
    arr = (ctypes.c_void_p * len(ps))(*[t.data_ptr() for t in ps])
    _call("mvip_mlp_pack_weights", arr, _ptr(out), _stream())
    return out


def _points_struct(rays=None, z_vals=None, viewdir_offset=8, pts=None, dirs=None):
    s = _lib.MvipPoints()
    keep = []
    if rays is not None:
        rays = _f32(rays, "rays")
        z_vals = _f32(z_vals, "z_vals")
        keep += [rays, z_vals]
        s.rays = rays.data_ptr()
        s.ray_stride = rays.shape[1]
        s.viewdir_offset = viewdir_offset
        s.z_vals = z_vals.data_ptr()
        s.n_rays = rays.shape[0]
        s.n_samples = z_vals.shape[1]
        s.n_points = rays.shape[0] * z_vals.shape[1]
    else:
        if pts.dtype != torch.float32 or dirs.dtype != torch.float32 or not pts.is_cuda:
            raise RuntimeError("pts/dirs must be fp32 CUDA tensors")
        if pts.stride(-1) != 1 or dirs.stride(-1) != 1:
            pts, dirs = pts.contiguous(), dirs.contiguous()
        keep += [pts, dirs]
        s.rays = None
        s.pts = pts.data_ptr()
        s.pts_stride = pts.stride(0)
        s.dirs = dirs.data_ptr()
        s.dirs_stride = dirs.stride(0)
        s.n_points = pts.shape[0]
    return s, keep


def mlp_forward(packed, rays=None, z_vals=None, viewdir_offset=8, pts=None, dirs=None, want_stash=False):
    """-> raw [P,4] (and the stash buffer when want_stash)"""
    lib = _lib.load()
    s, keep = _points_struct(rays, z_vals, viewdir_offset, pts, dirs)
    dev = keep[0].device
    raw = torch.empty((s.n_points, 4), device=dev, dtype=torch.float32)
    stash = _aligned_bytes(lib.mvip_mlp_stash_bytes(s.n_points), dev) if want_stash else None
    _call("mvip_mlp_forward", _ptr(packed), ctypes.byref(s), _ptr(raw), _ptr(stash), _stream())
    return (raw, stash) if want_stash else raw


class _GradArena:
    """Optional caller-owned buffer the flat gradient buffers of successive mlp_backward calls are carved from, back to back
    (fine network first, then coarse: autograd's order), so that the gradients of BOTH networks are one contiguous fp32 range
    and the data-parallel step needs ONE allreduce (dist.GradSync).  graph.GraphedTrainStep installs one per step."""

    def __init__(self):
        self.buf, self.off = None, 0

    def begin(self, buf):
        self.buf, self.off = buf, 0

    def end(self):
        self.buf, self.off = None, 0

    def take(self, n, dev, zero):
        if self.buf is None or self.buf.device != dev or self.off + n > self.buf.numel():
            return (torch.zeros if zero else torch.empty)((n,), device=dev, dtype=torch.float32)
        out = self.buf[self.off:self.off + n]
        self.off += n
        if zero:
            out.zero_()
        return out


grad_arena = _GradArena()


def mlp_backward(packed, d_raw, stash, grads=None, accumulate=False, want_workspace=False):
    """-> list of 24 fp32 gradient tensors in PARAM_ORDER (and the workspace holding this call's dZ images when
    want_workspace: what mlp_input_grad reads)"""
    lib = _lib.load()
    d_raw = _f32(d_raw, "d_raw").reshape(-1, 4)
    P = d_raw.shape[0]
    dev = d_raw.device
    if grads is None:
        # one flat buffer, 24 views
        sizes = [int(torch.Size(shp).numel()) for shp in PARAM_SHAPES]
        # the reduce kernel overwrites every element — except for an empty batch, which launches nothing
        flat = grad_arena.take(sum(sizes), dev, zero=(P == 0))
        grads, off = [], 0
        for shp, n in zip(PARAM_SHAPES, sizes):
            grads.append(flat[off:off + n].view(shp))
            off += n
        accumulate = False
    ws = _aligned_bytes(lib.mvip_mlp_backward_workspace_bytes(P), dev)
    arr = (ctypes.c_void_p * len(grads))(*[g.data_ptr() for g in grads])
    if kernel_timer.on:   # one bracket per launch: fused dgrad chain + weight gradients, head grads, reduce
        for bit, label in ((1, "backward_fused_kernel"), (4, "head_grads_kernel"), (8, "reduce_kernel")):
            _call(("mvip_mlp_backward_phases", label), _ptr(packed), _ptr(d_raw), P, _ptr(stash), _ptr(ws), arr,
                  int(bool(accumulate)), bit, _stream())
    else:
        _call("mvip_mlp_backward", _ptr(packed), _ptr(d_raw), P, _ptr(stash), _ptr(ws), arr, int(bool(accumulate)),
              _stream())
    return (grads, ws) if want_workspace else grads


def mlp_input_grad(packed, workspace, rays=None, z_vals=None, viewdir_offset=8, pts=None, dirs=None):
    """Gradient w.r.t. the MLP's inputs from the dZ images of the mlp_backward call that filled `workspace` (same points).
    -> d rays [N, ray_stride] (rays mode: o / d / viewdir columns, zeros elsewhere) or (d pts [P,3], d dirs [P,3])"""
    global launch_count
    s, keep = _points_struct(rays, z_vals, viewdir_offset, pts, dirs)
    dev = keep[0].device
    d6 = torch.empty((s.n_points, 6), device=dev, dtype=torch.float32)
    d_rays = torch.empty((s.n_rays, s.ray_stride), device=dev, dtype=torch.float32) if rays is not None else None
    _call("mvip_mlp_input_grad", _ptr(packed), ctypes.byref(s), _ptr(workspace), _ptr(d6), _ptr(d_rays), _stream())
    if rays is not None:
        launch_count += 1 if s.n_points > 0 else 0     # the per-ray sum is a second launch
        return d_rays
    return d6[:, 0:3], d6[:, 3:6]


def selftest_umma(which, a, b):
    a = _f32(a, "a")
    b = _f32(b, "b")
    if which == 0:
        K, N = a.shape[1], b.shape[0]
    else:
        K, N = a.shape[0], b.shape[1]
    out = torch.empty((128, N), device=a.device, dtype=torch.float32)
    _call("mvip_selftest_umma", int(which), _ptr(a), _ptr(b), N, K, _ptr(out), _stream())
    return out
