"""Drop-in for the render path of the reference's DS_NeRF/run.py:
batchify / run_network (:1096-1124), batchify_rays (:1127), render (:1143), create_nerf (:1474),
render_rays (:1703), depth2xyz_torch (:1909), depth2normal_geo (:1924).

Same names, arguments and return structures; the per-ray math runs in the sm_100a kernels of
libmvip_nerf.so.  The training driver, data loaders, SDS guidance, GUI and the tcnn model are out of scope
(SURVEY.md §2) and stay with the reference, which can import these functions in place of its own.
"""
import os

import numpy as np
import torch
import torch.nn as nn

from . import ops
from .dist import _flat_view
from .optim import FusedAdam
from .run_nerf_helpers import (NeRF, _NormalFromXYZ, get_embedder, get_rays, ndc_rays, raw2outputs, sample_pdf)

device = torch.device("cuda" if torch.cuda.is_available() else "cpu")
DEBUG = False


class DataParallel(nn.Module):
    """Stand-in for the nn.DataParallel wrapper of run.py:1491/1527: keeps the `module.` prefix of the
    reference's checkpoints (run.py:1043-1053) and the `.module` attribute, without the per-call
    scatter/broadcast/gather.  Scale-out is one process per GPU (mvip_nerf_b200.dist)."""

    def __init__(self, module, device_ids=None):
        super().__init__()
        self.module = module

    def forward(self, *a, **kw):
        return self.module(*a, **kw)


def _unwrap(net):
    return net.module if isinstance(net, (DataParallel, nn.DataParallel)) else net


def batchify(fn, chunk):
    """(run.py:1096-1105)"""
    if chunk is None:
        return fn

    def ret(inputs):
        return torch.cat([fn(inputs[i:i + chunk]) for i in range(0, inputs.shape[0], chunk)], 0)
    return ret


def run_network(inputs2, viewdirs, fn, embed_fn, embeddirs_fn, netchunk=1024 * 64):
    """(run.py:1108-1124) inputs2 [N,S,3], viewdirs [N,3] -> [N,S,4].

    When `fn` is our NeRF and the embedders are the standard ones, the embedding is never materialised: the
    fused kernel encodes on chip (netchunk is then irrelevant — the kernel is persistent and tiles internally).
    Otherwise the reference's sequence is followed with our embed kernel and `fn` applied in netchunk pieces."""
    net = _unwrap(fn)
    flat = torch.reshape(inputs2, [-1, inputs2.shape[-1]])
    fused = (isinstance(net, NeRF) and viewdirs is not None and getattr(embed_fn, "multires", None) == 10 and
             getattr(embeddirs_fn, "multires", None) == 4 and flat.shape[-1] == 3)
    if fused:
        dirs = viewdirs[:, None].expand(inputs2.shape).reshape(-1, 3)
        out = net.query_points(flat.contiguous(), dirs.contiguous())
        return torch.reshape(out, list(inputs2.shape[:-1]) + [4])
    embedded = embed_fn(flat)
    if viewdirs is not None:
        input_dirs = viewdirs[:, None].expand(inputs2.shape)
        embedded = torch.cat([embedded, embeddirs_fn(torch.reshape(input_dirs, [-1, input_dirs.shape[-1]]))], -1)
    outputs_flat = batchify(fn, netchunk)(embedded)
    return torch.reshape(outputs_flat, list(inputs2.shape[:-1]) + [outputs_flat.shape[-1]])


class _FusedQuery:
    """network_query_fn built by create_nerf: callable like the reference's closure (run.py:1530-1533) and
    recognised by render_rays, which then feeds rays + depths straight to the fused kernel."""

    def __init__(self, embed_fn, embeddirs_fn, netchunk):
        self.embed_fn, self.embeddirs_fn, self.netchunk = embed_fn, embeddirs_fn, netchunk

    def __call__(self, inputs, viewdirs, network_fn):
        return run_network(inputs, viewdirs, network_fn, embed_fn=self.embed_fn, embeddirs_fn=self.embeddirs_fn,
                           netchunk=self.netchunk)


def batchify_rays(rays_flat, chunk=1024 * 32, need_alpha=False, detach_weights=False, _mse=None, **kwargs):
    """(run.py:1127-1140) render in chunks, concatenate per key.  `_mse=(target_rgb | None, target_disp | None)` (ours): per-ray
    targets of the fused photometric losses, chunked with the rays; the squared-error sums `sqerr` / `sqerr0` are added up."""
    pieces = {}
    for i in range(0, rays_flat.shape[0], chunk):
        mse = None if _mse is None else tuple(None if t is None else t.reshape(rays_flat.shape[0], -1)[i:i + chunk] for t in _mse)
        ret = render_rays(rays_flat[i:i + chunk], need_alpha=need_alpha, detach_weights=detach_weights, _mse=mse, **kwargs)
        for k, v in ret.items():
            pieces.setdefault(k, []).append(v)
    out = {}
    for k, v in pieces.items():
        if k in ("sqerr", "sqerr0"):
            out[k] = v[0] if len(v) == 1 else torch.stack(v, 0).sum(0)
        else:
            out[k] = v[0] if len(v) == 1 else torch.cat(v, 0)
    return out


def _is_number(x):
    return isinstance(x, (int, float)) or (isinstance(x, np.generic) and np.ndim(x) == 0)


def _clip_patch(patch, H, W):
    """(i, j, len1, len2) clipped to the image the way the reference's slicing rays_o[i:i+len1, j:j+len2] clips (run.py:1174)."""
    i, j, len1, len2 = [int(v) for v in patch]
    i, j = max(0, min(i, H)), max(0, min(j, W))
    return i, j, max(0, min(i + len1, H) - i), max(0, min(j + len2, W) - j)


def _pose_tensor(x, dev=None):
    """[3,4] fp32 CUDA view of a pose (numpy or tensor); differentiable torch ops, so a pose that requires grad stays in the graph"""
    t = torch.as_tensor(x, dtype=torch.float32)
    dev = dev or (t.device if t.is_cuda else torch.device("cuda", torch.cuda.current_device()))
    return t.to(dev)[:3, :4].contiguous()


class _RaysFromPose(torch.autograd.Function):
    """ops.rays_from_pose with its backward kernel: d batch -> d c2w (and d c2w_staticcam)"""

    @staticmethod
    def forward(ctx, c2w, c2w_staticcam, H, W, focal, near, far, use_viewdirs, window, ndc):
        ctx.save_for_backward(c2w, c2w_staticcam)
        ctx.cam = (H, W, focal, window, use_viewdirs, ndc)
        return ops.rays_from_pose(H, W, focal, c2w, near, far, use_viewdirs=use_viewdirs, c2w_staticcam=c2w_staticcam,
                                  patch=window, ndc=ndc)

    @staticmethod
    def backward(ctx, g):
        c2w, cs = ctx.saved_tensors
        H, W, focal, window, use_viewdirs, ndc = ctx.cam
        g_c, g_cs = ops.rays_from_pose_backward(c2w, cs, H, W, focal, window or (0, 0, H, W), g, use_viewdirs=use_viewdirs, ndc=ndc)
        return (g_c, g_cs) + (None,) * 8


class _RaysFromPoses(torch.autograd.Function):
    """ops.rays_from_poses with its backward kernel: d batch -> d poses [V,3,4]"""

    @staticmethod
    def forward(ctx, poses, pixels, H, W, focal, near, far, use_viewdirs, ndc):
        ctx.save_for_backward(poses, pixels)
        ctx.cam = (H, W, focal, use_viewdirs, ndc)
        return ops.rays_from_poses(H, W, focal, poses, pixels, near, far, use_viewdirs=use_viewdirs, ndc=ndc)

    @staticmethod
    def backward(ctx, g):
        poses, pixels = ctx.saved_tensors
        H, W, focal, use_viewdirs, ndc = ctx.cam
        return (ops.rays_from_poses_backward(poses, pixels, H, W, focal, g, use_viewdirs=use_viewdirs, ndc=ndc),) + (None,) * 8


class _RaysPack(torch.autograd.Function):
    """ops.rays_pack with its backward kernel: d batch -> d rays_o, d rays_d"""

    @staticmethod
    def forward(ctx, rays_o, rays_d, near, far, use_viewdirs, ndc, H, W, focal):
        ctx.save_for_backward(rays_o, rays_d)
        ctx.cam = (use_viewdirs, ndc, H, W, focal)
        return ops.rays_pack(rays_o, rays_d, near, far, use_viewdirs=use_viewdirs, ndc=ndc, H=H, W=W, focal=focal)

    @staticmethod
    def backward(ctx, g):
        rays_o, rays_d = ctx.saved_tensors
        use_viewdirs, ndc, H, W, focal = ctx.cam
        g_o, g_d, _ = ops.rays_pack_backward(rays_o, rays_d, None, g, use_viewdirs=use_viewdirs, ndc=ndc, H=H, W=W, focal=focal)
        return (g_o.view(rays_o.shape), g_d.view(rays_d.shape)) + (None,) * 7


def _needs_grad(*xs):
    return torch.is_grad_enabled() and any(torch.is_tensor(x) and x.requires_grad for x in xs)


def _pose_table_rays(H, W, focal, c2w, pixels, rays, ndc, near, far, use_viewdirs, c2w_staticcam, depths, patch):
    """The `pixels=` form of the ray-batch assembly: c2w [V,3,4] | [V,4,4], pixels [N,3] = (view, row, col) -> ([N, 8|11], sh)"""
    if c2w is None or rays is not None or c2w_staticcam is not None or depths is not None or patch is not None:
        raise ValueError("pixels= takes a pose stack c2w [V,3,4] and no rays / c2w_staticcam / depths / patch")
    if not (_is_number(near) and _is_number(far) and _is_number(focal)):
        raise NotImplementedError("pixels=: near, far and focal must be scalars (the pose-table ray kernel takes scalars)")
    t = torch.as_tensor(c2w, dtype=torch.float32)
    dev = t.device if t.is_cuda else torch.device("cuda", torch.cuda.current_device())
    if t.dim() != 3:
        raise ValueError("pixels= needs a pose stack c2w [V,3,4] or [V,4,4], got %s" % (tuple(t.shape),))
    poses = t.to(dev)[:, :3, :4].contiguous()
    pixels = torch.as_tensor(pixels, device=dev)
    if _needs_grad(poses):
        rays_flat = _RaysFromPoses.apply(poses, pixels, H, W, focal, near, far, use_viewdirs, ndc)
    else:
        rays_flat = ops.rays_from_poses(H, W, focal, poses, pixels, near, far, use_viewdirs=use_viewdirs, ndc=ndc)
    return rays_flat, (pixels.shape[0], 3)


def _assemble_rays(H, W, focal, rays, c2w, ndc, near, far, use_viewdirs, c2w_staticcam, depths, patch, pixels=None):
    """The ray-batch assembly of render() (run.py:1171-1207) -> (rays_flat [N, 8|9|11|12], sh).

    The batch is written by ONE kernel (get_rays / patch / viewdir normalisation / ndc_rays / near / far / cat):
    mvip_rays_from_pose for `c2w=`, mvip_rays_pack for `rays=`.  Only the `depths=` column (used by the out-of-scope sigma
    loss), non-scalar near / far / focal and `rays=` combined with a static camera take the elementwise torch route.
    When the pose(s) or the given rays require grad, the fused entries run inside autograd Functions whose backward kernels
    return d c2w / d c2w_staticcam or d rays_o / d rays_d; the torch route is differentiable as it stands.
    With `pixels` [N,3] = (view, row, col), c2w is a pose stack and mvip_rays_from_poses writes the batch (d stack when it
    requires grad)."""
    if pixels is not None:
        return _pose_table_rays(H, W, focal, c2w, pixels, rays, ndc, near, far, use_viewdirs, c2w_staticcam, depths, patch)
    fusable = depths is None and torch.cuda.is_available() and _is_number(near) and _is_number(far) and _is_number(focal)
    if fusable and c2w is not None:
        if patch is not None:
            patch = _clip_patch(patch, H, W)
        if _needs_grad(c2w, c2w_staticcam):
            c = _pose_tensor(c2w)
            cs = None if c2w_staticcam is None else _pose_tensor(c2w_staticcam, c.device)
            rays_flat = _RaysFromPose.apply(c, cs, H, W, focal, near, far, use_viewdirs, patch, ndc)
        else:
            rays_flat = ops.rays_from_pose(H, W, focal, c2w, near, far, use_viewdirs=use_viewdirs, c2w_staticcam=c2w_staticcam,
                                           patch=patch, ndc=ndc)
        return rays_flat, ((H, W) if patch is None else (patch[2], patch[3])) + (3,)
    if fusable and c2w is None and (c2w_staticcam is None or not use_viewdirs):
        rays_o, rays_d = rays
        if _needs_grad(rays_o, rays_d):
            return _RaysPack.apply(rays_o, rays_d, near, far, use_viewdirs, ndc, H, W, focal), rays_d.shape
        return ops.rays_pack(rays_o, rays_d, near, far, use_viewdirs=use_viewdirs, ndc=ndc, H=H, W=W, focal=focal), rays_d.shape
    if c2w is not None:
        rays_o, rays_d = get_rays(H, W, focal, c2w)
        if patch is not None:
            i, j, len1, len2 = patch
            rays_o = rays_o[i:i + len1, j:j + len2, :]
            rays_d = rays_d[i:i + len1, j:j + len2, :]
    else:
        rays_o, rays_d = rays
    viewdirs = None
    if use_viewdirs:
        viewdirs = rays_d
        if c2w_staticcam is not None:
            rays_o, rays_d = get_rays(H, W, focal, c2w_staticcam)
        viewdirs = viewdirs / torch.norm(viewdirs, dim=-1, keepdim=True)
        viewdirs = torch.reshape(viewdirs, [-1, 3]).float()
    sh = rays_d.shape
    if ndc:
        rays_o, rays_d = ndc_rays(H, W, focal, 1., rays_o, rays_d)
    rays_o = torch.reshape(rays_o, [-1, 3]).float()
    rays_d = torch.reshape(rays_d, [-1, 3]).float()
    ones = torch.ones_like(rays_d[..., :1])
    cols = [rays_o, rays_d, near * ones, far * ones]
    if depths is not None:
        cols.append(depths.reshape(-1, 1).to(rays_d))
    if use_viewdirs:
        cols.append(viewdirs)
    return torch.cat(cols, -1), sh


def _split_outputs(all_ret, sh):
    for k in all_ret:
        if k not in ("sqerr", "sqerr0"):           # per-batch sums of the fused losses: not one row per ray
            all_ret[k] = torch.reshape(all_ret[k], list(sh[:-1]) + list(all_ret[k].shape[1:]))
    k_extract = ['rgb_map', 'disp_map', 'acc_map', 'depth_map']
    return [all_ret[k] for k in k_extract] + [{k: all_ret[k] for k in all_ret if k not in k_extract}]


def render(H, W, focal, chunk=1024 * 32, rays=None, c2w=None, ndc=True, near=0., far=1., use_viewdirs=False,
           c2w_staticcam=None, depths=None, need_alpha=False, detach_weights=False, patch=None, pixels=None, **kwargs):
    """(run.py:1143-1219) -> [rgb_map, disp_map, acc_map, depth_map, extras].
    `pixels` (ours) [N,3] int = (view, row, col): c2w is then a pose stack [V,3,4] | [V,4,4], the batch is those N pixels of
    their views (a training batch drawn from many views, run.py:889-908), the maps are [N, ...], and a stack that requires grad
    gets d stack."""
    rays_flat, sh = _assemble_rays(H, W, focal, rays, c2w, ndc, near, far, use_viewdirs, c2w_staticcam, depths, patch, pixels)
    all_ret = batchify_rays(rays_flat, chunk, need_alpha=need_alpha, detach_weights=detach_weights, **kwargs)
    return _split_outputs(all_ret, sh)


def create_nerf(args):
    """(run.py:1474-1599) -> (render_kwargs_train, render_kwargs_test, start, grad_vars, optimizer)."""
    embed_fn, input_ch = get_embedder(args.multires, args.i_embed)
    input_ch_views, embeddirs_fn = 0, None
    if args.use_viewdirs:
        embeddirs_fn, input_ch_views = get_embedder(args.multires_views, args.i_embed)
    if getattr(args, "alpha_model_path", None) is not None:
        raise NotImplementedError("alpha_model_path / NeRF_RGB is out of scope (unused by config_1, run.py:173)")
    output_ch = 5 if args.N_importance > 0 else 4
    skips = [4]
    dev = torch.device("cuda", torch.cuda.current_device()) if torch.cuda.is_available() else torch.device("cpu")
    model = DataParallel(NeRF(D=args.netdepth, W=args.netwidth, input_ch=input_ch, output_ch=output_ch, skips=skips,
                              input_ch_views=input_ch_views, use_viewdirs=args.use_viewdirs).to(dev))
    grad_vars = list(model.parameters())
    model_fine = None
    if args.N_importance > 0:
        model_fine = NeRF(D=args.netdepth_fine, W=args.netwidth_fine, input_ch=input_ch, output_ch=output_ch,
                          skips=skips, input_ch_views=input_ch_views, use_viewdirs=args.use_viewdirs).to(dev)
        grad_vars += list(model_fine.parameters())
        model_fine = DataParallel(model_fine)

    network_query_fn = _FusedQuery(embed_fn, embeddirs_fn, args.netchunk)
    optimizer = FusedAdam(params=grad_vars, lr=args.lrate, betas=(0.9, 0.999))   # torch.optim.Adam semantics, one launch per step

    start = 0
    basedir, expname = args.basedir, args.expname
    if args.ft_path is not None and args.ft_path != 'None':
        ckpts = [args.ft_path]
    else:
        d = os.path.join(basedir, expname)
        ckpts = [os.path.join(d, f) for f in sorted(os.listdir(d)) if 'tar' in f]
    print('Found ckpts', ckpts)
    if len(ckpts) > 0 and not args.no_reload:
        ckpt_path = ckpts[-1]
        print('Reloading from', ckpt_path)
        ckpt = torch.load(ckpt_path, map_location=dev)
        start = ckpt['global_step']
        optimizer.load_state_dict(ckpt['optimizer_state_dict'])
        model.load_state_dict(ckpt['network_fn_state_dict'])
        if model_fine is not None:
            model_fine.load_state_dict(ckpt['network_fine_state_dict'])

    render_kwargs_train = {
        'network_query_fn': network_query_fn, 'perturb': args.perturb, 'N_importance': args.N_importance,
        'network_fine': model_fine, 'N_samples': args.N_samples, 'network_fn': model,
        'use_viewdirs': args.use_viewdirs, 'white_bkgd': args.white_bkgd, 'raw_noise_std': args.raw_noise_std,
    }
    if args.dataset_type != 'llff' or args.no_ndc:
        print('Not ndc!')
        render_kwargs_train['ndc'] = False
        render_kwargs_train['lindisp'] = args.lindisp
    else:
        render_kwargs_train['ndc'] = True
    render_kwargs_test = dict(render_kwargs_train)
    render_kwargs_test['perturb'] = False
    render_kwargs_test['raw_noise_std'] = 0.
    if getattr(args, "sigma_loss", False):
        raise NotImplementedError("SigmaLoss (loss.py) is out of scope: unset in config_1 (SURVEY.md §2 row 13)")
    return render_kwargs_train, render_kwargs_test, start, grad_vars, optimizer


def _pytest_uniform(shape, dev):
    np.random.seed(0)
    return torch.Tensor(np.random.rand(*list(shape))).to(dev)


def render_rays(ray_batch, network_fn, network_query_fn, N_samples, retraw=False, lindisp=False, perturb=0.,
                N_importance=0, network_fine=None, white_bkgd=False, raw_noise_std=0., pytest=False, sigma_loss=None,
                verbose=False, need_alpha=False, detach_weights=False, _randoms=None, _mse=None):
    """(run.py:1703-1847) volumetric rendering of one chunk of rays -> dict with the reference's keys.

    Random numbers are drawn on the host side in the reference's order (t_rand, coarse noise, u, fine noise)
    and handed to the kernels; `_randoms` (dict with any of t_rand / noise0 / u / noise1) overrides them so
    tests and multi-GPU runs can share one stream."""
    if network_fn is None:
        raise NotImplementedError("render_rays without a coarse network (alpha_model path) is out of scope")
    if sigma_loss is not None:
        raise NotImplementedError("sigma_loss is out of scope (SURVEY.md §2 row 13)")
    rnd = _randoms or {}
    ray_batch = ray_batch.float().contiguous()
    dev = ray_batch.device
    N_rays = ray_batch.shape[0]
    rays_d = ray_batch[:, 3:6]
    has_dirs = ray_batch.shape[-1] > 9
    coarse = _unwrap(network_fn)
    fused = isinstance(network_query_fn, _FusedQuery) and isinstance(coarse, NeRF) and has_dirs

    # ---- stratified samples (run.py:1759-1781) --------------------------------------------------------
    t_vals = torch.linspace(0., 1., steps=N_samples, device=dev)
    t_rand = None
    if perturb > 0.:
        t_rand = rnd.get("t_rand")
        if t_rand is None:
            t_rand = _pytest_uniform((N_rays, N_samples), dev) if pytest else torch.rand((N_rays, N_samples), device=dev)
    z_vals = ops.sample_coarse(ray_batch, t_vals, t_rand, lindisp)

    def query(net, z):
        if fused and isinstance(_unwrap(net), NeRF):
            return _unwrap(net).query_rays(ray_batch, z)
        pts = ray_batch[:, None, 0:3] + ray_batch[:, None, 3:6] * z[..., :, None]
        return network_query_fn(pts, ray_batch[:, -3:] if has_dirs else None, net)

    def noise_for(shape, key):
        if key in rnd:
            return rnd[key]
        if raw_noise_std > 0.:
            if pytest:
                return _pytest_uniform(shape, dev) * raw_noise_std
            n = torch.randn(shape, device=dev)
            return n if raw_noise_std == 1. else n * raw_noise_std     # x * 1.0 == x: skip the launch
        return None

    raw = query(network_fn, z_vals)
    rgb_map, disp_map, acc_map, weights, depth_map, alpha, *sq = raw2outputs(
        raw, z_vals, rays_d, raw_noise_std, white_bkgd, need_alpha=need_alpha, detach_weights=detach_weights,
        _noise=noise_for((N_rays, N_samples), "noise0"), _mse=_mse)

    z_std = None
    if N_importance > 0:
        rgb_map_0, disp_map_0, acc_map_0, alpha0, sq0 = rgb_map, disp_map, acc_map, alpha, sq
        # ---- hierarchical samples: z_mid, sample_pdf, detach, sort-merge (run.py:1809-1816) ------------
        u = rnd.get("u")
        if u is None:
            if perturb == 0.:
                u = torch.linspace(0., 1., steps=N_importance, device=dev)
                if pytest:
                    u = torch.Tensor(np.linspace(0., 1., N_importance)).to(dev)
            else:
                u = _pytest_uniform((N_rays, N_importance), dev) if pytest else torch.rand((N_rays, N_importance), device=dev)
        fs = ops.sample_fine(z_vals, weights.detach(), u, want_samples=False)
        z_vals, z_std = fs["z_merged"], fs["z_std"]
        run_fn = network_fn if network_fine is None else network_fine
        raw = query(run_fn, z_vals)
        rgb_map, disp_map, acc_map, weights, depth_map, alpha, *sq = raw2outputs(
            raw, z_vals, rays_d, raw_noise_std, white_bkgd, need_alpha=need_alpha, detach_weights=detach_weights,
            _noise=noise_for((N_rays, N_samples + N_importance), "noise1"), _mse=_mse)

    ret = {'rgb_map': rgb_map, 'disp_map': disp_map, 'acc_map': acc_map, 'depth_map': depth_map,
           'weights': weights, 'z_vals': z_vals}
    if retraw:
        ret['raw'] = raw
    if need_alpha:
        ret['alpha'] = alpha
        ret['alpha0'] = alpha0      # NameError when N_importance == 0, exactly as in the reference (run.py:1831)
    if N_importance > 0:
        ret['rgb0'] = rgb_map_0
        ret['disp0'] = disp_map_0
        ret['acc0'] = acc_map_0
        ret['z_std'] = z_std
    if _mse is not None:             # fused img2mse: [sum (rgb - target)^2, sum (disp - target)^2] of the fine / coarse maps
        ret['sqerr'] = sq[0]
        if N_importance > 0:
            ret['sqerr0'] = sq0[0]
    if DEBUG:
        for k in ret:
            if torch.isnan(ret[k]).any() or torch.isinf(ret[k]).any():
                print(f"! [Numerical Error] {k} contains nan or inf.")
    return ret


# ---------------------------------------------------------------------------------------------------
# deferred back-propagation (SURVEY.md §8 f2): full guidance views with gradients in bounded memory
# ---------------------------------------------------------------------------------------------------
_DIFF_KEYS = ("rgb_map", "disp_map", "acc_map", "depth_map", "rgb0", "disp0", "acc0")


def _net_params(render_kwargs):
    """[(net, ordered parameter list)] of the coarse / fine networks of a render-kwargs dict."""
    nets = []
    for key in ("network_fn", "network_fine"):
        net = render_kwargs.get(key)
        if net is not None:
            net = _unwrap(net)
            nets.append((net, net._ordered_params() if isinstance(net, NeRF) else list(net.parameters())))
    return nets


class _DeferredRays(torch.autograd.Function):
    """rays_flat -> the integrated maps of batchify_rays, WITHOUT keeping any per-sample state for the backward pass.

    forward  renders every chunk under no_grad (no activation stash: the tensor-bound render kernel);
    backward re-renders one chunk at a time with the stash enabled, back-propagates the slice of the upstream image
             gradients that belongs to it and accumulates the parameter gradients; when rays_flat requires grad (a pose or rays
             that require grad upstream), each chunk's slice is a grad leaf and the slices' gradients are concatenated.
    Peak memory is one chunk's stash (10.3 KB per sample point) instead of the whole view's: 4 x 512 x 512 rays x 192 points
    would need 2 TB, which is why the reference cannot run its guidance views at normalmap_render_factor = 1 (README.md:61).
    The random streams (perturb / raw_noise_std) are replayed by restoring the CUDA generator state, so the re-rendered
    chunks are the ones the loss saw."""

    @staticmethod
    def forward(ctx, rays_flat, chunk, kw, holder, *params):
        dev = rays_flat.device
        ctx.rng = torch.cuda.get_rng_state(dev) if dev.type == "cuda" else torch.get_rng_state()
        ret = batchify_rays(rays_flat, chunk, **kw)
        keys = list(ret.keys())
        holder["keys"] = keys
        ctx.keys, ctx.chunk, ctx.kw, ctx.rays = keys, chunk, kw, rays_flat
        ctx.params = params
        ctx.set_materialize_grads(False)
        outs = tuple(ret[k] for k in keys)
        ctx.mark_non_differentiable(*[ret[k] for k in keys if k not in _DIFF_KEYS])
        return outs

    @staticmethod
    def backward(ctx, *gouts):
        grads = {k: g for k, g in zip(ctx.keys, gouts) if g is not None and k in _DIFF_KEYS}
        none = (None,) * (4 + len(ctx.params))
        if not grads:
            return none
        params = [p for p in ctx.params]
        live = [i for i, p in enumerate(params) if p.requires_grad]
        want_rays = ctx.needs_input_grad[0]
        if not live and not want_rays:
            return none
        d_rays = []
        dev = ctx.rays.device
        acc = [None] * len(params)
        flat_acc = {}            # first parameter index of a network -> (flat accumulator, its per-parameter views)
        with torch.random.fork_rng(devices=[dev] if dev.type == "cuda" else []):
            if dev.type == "cuda":
                torch.cuda.set_rng_state(ctx.rng, dev)
            else:
                torch.set_rng_state(ctx.rng)
            for i in range(0, ctx.rays.shape[0], ctx.chunk):
                with torch.enable_grad():
                    rays = ctx.rays[i:i + ctx.chunk].detach().requires_grad_(want_rays)
                    ret = render_rays(rays, **ctx.kw)
                    outs = [ret[k] for k in grads]
                    gs = [grads[k][i:i + ctx.chunk].contiguous() for k in grads]
                    wrt = [params[j] for j in live] + ([rays] if want_rays else [])
                    got = torch.autograd.grad(outs, wrt, gs, allow_unused=True)
                    g = dict(zip(live, got[:len(live)]))
                    if want_rays:
                        d_rays.append(torch.zeros_like(rays) if got[-1] is None else got[-1])
                for a in range(0, len(params), len(ops.PARAM_ORDER)):
                    # the MLP backward writes a network's 24 gradients back to back: accumulate them as ONE tensor
                    idx = list(range(a, min(a + len(ops.PARAM_ORDER), len(params))))
                    gl = [g.get(j) for j in idx]
                    flat = _flat_view(gl) if all(x is not None for x in gl) else None
                    if flat is not None and (a in flat_acc or all(acc[j] is None for j in idx)):
                        if a not in flat_acc:
                            buf = flat.clone()
                            views, off = [], 0
                            for x in gl:
                                views.append(buf[off:off + x.numel()].view(x.shape))
                                off += x.numel()
                            flat_acc[a] = buf
                            for j, v in zip(idx, views):
                                acc[j] = v
                        else:
                            flat_acc[a].add_(flat)
                        continue
                    for j, gj in zip(idx, gl):
                        if gj is not None:
                            acc[j] = gj.clone() if acc[j] is None else acc[j].add_(gj)
        return (torch.cat(d_rays, 0) if want_rays else None, None, None, None) + tuple(acc)


def render_deferred(H, W, focal, chunk=1024 * 8, rays=None, c2w=None, ndc=True, near=0., far=1., use_viewdirs=False,
                    c2w_staticcam=None, depths=None, need_alpha=False, detach_weights=False, patch=None, pixels=None, **kwargs):
    """render() with deferred back-propagation: same arguments (pixels= included) and return list; rgb / disp / acc / depth (+ rgb0 /
    disp0 / acc0) carry gradients to the network parameters and, when c2w / c2w_staticcam / rays require grad, to them; the per-sample extras
    (weights, z_vals, raw, alpha) are detached.
    `chunk` is the number of rays whose activations exist at any one time during backward (default 8192: 16 GB)."""
    if depths is not None:
        raise NotImplementedError("render_deferred: the depths column (sigma loss) is out of scope")
    rays_flat, sh = _assemble_rays(H, W, focal, rays, c2w, ndc, near, far, use_viewdirs, c2w_staticcam, None, patch, pixels)
    kw = dict(kwargs, need_alpha=need_alpha, detach_weights=detach_weights)
    params = [p for _, ps in _net_params(kwargs) for p in ps]
    holder = {}
    outs = _DeferredRays.apply(rays_flat, int(chunk), kw, holder, *params)
    return _split_outputs(dict(zip(holder["keys"], outs)), sh)


# ---------------------------------------------------------------------------------------------------
# view loops (run.py:1222-1432): render_path / render_path_4view / render_path_projection
# ---------------------------------------------------------------------------------------------------
def _write_png(path, img8):
    """8-bit RGB / grey PNG without imageio (absent in this image): zlib + the four mandatory chunks."""
    import struct
    import zlib
    a = np.ascontiguousarray(img8, dtype=np.uint8)
    if a.ndim == 2:
        a = a[..., None]
    h, w, c = a.shape
    ctype = {1: 0, 3: 2, 4: 6}[c]
    rows = np.concatenate([np.zeros((h, 1), np.uint8), a.reshape(h, w * c)], 1).tobytes()

    def chunk(tag, data):
        return struct.pack(">I", len(data)) + tag + data + struct.pack(">I", zlib.crc32(tag + data) & 0xffffffff)
    with open(path, "wb") as f:
        f.write(b"\x89PNG\r\n\x1a\n" + chunk(b"IHDR", struct.pack(">IIBBBBB", w, h, 8, ctype, 0, 0, 0)) +
                chunk(b"IDAT", zlib.compress(rows, 6)) + chunk(b"IEND", b""))


def _imwrite(path, img8):
    try:
        import imageio
        imageio.imwrite(path, img8)
    except Exception:
        _write_png(path, img8)


def _scaled_hwf(hwf, render_factor):
    H, W, focal = hwf
    if render_factor != 0:
        H, W, focal = H // render_factor, W // render_factor, focal / render_factor
    K = np.array([[focal, 0, W / 2], [0, focal, H / 2], [0, 0, 1]])
    return int(H), int(W), focal, K


def render_path(render_poses, hwf, chunk, render_kwargs, gt_imgs=None, savedir=None, render_factor=0,
                disp_require_grad=False, need_alpha=False, rgb_require_grad=False, detach_weights=False,
                patch_len=None, masks=None, deferred_backprop=False):
    """(run.py:1222-1362) renders every pose; -> (rgbs, disps, (Xs, Ys)); with `savedir` writes the reference's layout
    (intrinsics.txt, rgb/*.png, depth|disp|weight|z|alpha/*.npy, pose/*.txt).  `deferred_backprop` (ours) renders the
    gradient-carrying views through render_deferred so that whole views fit in memory."""
    import random
    to8b = lambda x: (255 * np.clip(x, 0, 1)).astype(np.uint8)  # noqa: E731
    H, W, focal, K = _scaled_hwf(hwf, render_factor)
    if savedir is not None:
        np.savetxt(os.path.join(savedir, 'intrinsics.txt'), K)
    rgbs, disps, Xs, Ys = [], [], [], []
    for i, c2w in enumerate(render_poses):
        if disp_require_grad or rgb_require_grad:
            patch = None
            if patch_len is not None:
                masked = np.where(masks[i] != 0)
                masked = (masked[0] // render_factor, masked[1] // render_factor)
                Xs.append(random.randint(masked[0].min(), max(masked[0].max() - patch_len[0], masked[0].min())))
                Ys.append(random.randint(masked[1].min(), max(masked[1].max() - patch_len[1], masked[1].min())))
                patch = (Xs[-1], Ys[-1], patch_len[0], patch_len[1])
            fn = render_deferred if deferred_backprop else render
            rgb, disp, acc, depth, extras = fn(H, W, focal, chunk=chunk, c2w=c2w[:3, :4], retraw=True, need_alpha=need_alpha,
                                               detach_weights=detach_weights, patch=patch, **render_kwargs)
        else:
            with torch.no_grad():
                rgb, disp, acc, depth, extras = render(H, W, focal, chunk=chunk, c2w=c2w[:3, :4], retraw=True,
                                                       need_alpha=need_alpha, **render_kwargs)
        disps.append(disp if disp_require_grad else disp.detach().cpu().numpy())
        rgbs.append(rgb if rgb_require_grad else rgb.detach().cpu().numpy())
        if savedir is not None:
            dirs = {k: os.path.join(savedir, k) for k in ('rgb', 'depth', 'disp', 'weight', 'images', 'z', 'pose')}
            if need_alpha:
                dirs['alpha'] = os.path.join(savedir, 'alpha')
            for d in dirs.values():
                os.makedirs(d, exist_ok=True)
            rgb_np = rgbs[-1] if isinstance(rgbs[-1], np.ndarray) else rgbs[-1].detach().cpu().numpy()
            rgb8 = to8b(np.nan_to_num(rgb_np, nan=0.0))
            _imwrite(os.path.join(dirs['rgb'], '{:06d}.png'.format(i)), rgb8)
            if gt_imgs is not None:
                gt = gt_imgs[i]
                gt = gt.detach().cpu().numpy() if torch.is_tensor(gt) else np.asarray(gt)
                _imwrite(os.path.join(dirs['images'], '{:06d}.png'.format(i)), to8b(gt))
            np.save(os.path.join(dirs['depth'], '{:06d}.npy'.format(i)), depth.detach().cpu().numpy())
            np.save(os.path.join(dirs['disp'], '{:06d}.npy'.format(i)), disp.detach().cpu().numpy())
            np.save(os.path.join(dirs['weight'], '{:06d}.npy'.format(i)), extras['weights'].detach().cpu().numpy())
            np.save(os.path.join(dirs['z'], '{:06d}.npy'.format(i)), extras['z_vals'].detach().cpu().numpy())
            if need_alpha:
                np.save(os.path.join(dirs['alpha'], '{:06d}.npy'.format(i)), extras['alpha'].detach().cpu().numpy())
            pose = torch.as_tensor(render_poses[i])[:3, :4].detach().cpu().numpy()
            np.savetxt(os.path.join(dirs['pose'], '{:06d}.txt'.format(i)), np.concatenate([pose, np.array([[0, 0, 0, 1]])], 0))
    disps = torch.stack(disps, 0) if disp_require_grad else np.stack(disps, 0)
    rgbs = torch.stack(rgbs, 0) if rgb_require_grad else np.stack(rgbs, 0)
    return rgbs, disps, (Xs, Ys)


def render_path_4view(iter, all_masks, render_poses, hwf, chunk, render_kwargs, gt_imgs=None, savedir=None, render_factor=0,
                      disp_require_grad=False, need_alpha=False, rgb_require_grad=False, detach_weights=False,
                      patch_len=None, masks=None, deferred_backprop=False):
    """(run.py:1365-1402) collaborative-guidance views: every second pose of the +-4 neighbourhood of pose `iter % 60`,
    rendered WITH gradients -> (rgbs [V,H,W,3], disps [V,H,W], selected_masks)."""
    H, W, focal, _ = _scaled_hwf(hwf, render_factor)
    neighborhood_size = 4
    iter = iter % 60
    sel = slice(max(0, iter - neighborhood_size), min(len(render_poses), iter + neighborhood_size + 1), 2)
    selected_poses, selected_masks = render_poses[sel], all_masks[sel]
    fn = render_deferred if deferred_backprop else render
    rgbs, disps = [], []
    for c2w in selected_poses:
        rgb, disp, _, _, _ = fn(H, W, focal, chunk=chunk, c2w=c2w[:3, :4], retraw=True, need_alpha=need_alpha, **render_kwargs)
        disps.append(disp)
        rgbs.append(rgb)
    return torch.stack(rgbs, 0), torch.stack(disps, 0), selected_masks


def convert_pose(C2W):
    """(run.py:1435-1440)"""
    flip_yz = np.eye(4)
    flip_yz[1, 1] = -1
    flip_yz[2, 2] = -1
    return np.matmul(C2W, flip_yz)


def render_path_projection(render_poses, hwf, chunk, render_kwargs, render_factor=0):
    """(run.py:1405-1432) -> (z_vals, weights, c2ws, K) per pose, numpy."""
    H, W, focal, K = _scaled_hwf(hwf, render_factor)
    z_vals, weights, c2ws = [], [], []
    for i, c2w in enumerate(render_poses):
        with torch.no_grad():
            _, _, _, _, extras = render(H, W, focal, chunk=chunk, c2w=c2w[:3, :4], retraw=True, **render_kwargs)
        z_vals.append(extras['z_vals'].cpu().numpy())
        weights.append(extras['weights'].cpu().numpy())
        pose = torch.as_tensor(render_poses[i])[:3, :4].detach().cpu().numpy()
        c2ws.append(convert_pose(np.concatenate([pose, np.array([[0, 0, 0, 1]])], axis=0)))
    return z_vals, weights, c2ws, K


def save_checkpoint(path, global_step, render_kwargs_train, optimizer):
    """The `.tar` the reference's train() writes (run.py:1043-1053): same keys, `module.`-prefixed state dicts; create_nerf
    (ours or the reference's) reloads it."""
    torch.save({
        'global_step': global_step,
        'network_fn_state_dict': render_kwargs_train['network_fn'].state_dict()
        if render_kwargs_train['network_fn'] is not None else None,
        'network_fine_state_dict': render_kwargs_train['network_fine'].state_dict()
        if render_kwargs_train['network_fine'] is not None else None,
        'optimizer_state_dict': optimizer.state_dict(),
    }, path)


def update_learning_rate(optimizer, args, global_step):
    """(run.py:1031-1039) exponential decay, 0.1 every lrate_decay*1000 steps."""
    new_lrate = args.lrate * (0.1 ** (global_step / (args.lrate_decay * 1000)))
    for param_group in optimizer.param_groups:
        param_group['lr'] = new_lrate
    return new_lrate


# ---------------------------------------------------------------------------------------------------
# normal map from depth (run.py:1909-1940; call site :948-965)
# ---------------------------------------------------------------------------------------------------
def depth2xyz_torch(depth_map, depth_cam_matrix, depth_scale=1.0):
    """tensor(h,w), tensor(3,3) -> tensor(h,w,3)  (elementwise glue; the fused route is run_nerf_helpers.depth2normal)"""
    fx, fy = depth_cam_matrix[0, 0], depth_cam_matrix[1, 1]
    cx, cy = depth_cam_matrix[0, 2], depth_cam_matrix[1, 2]
    hh, ww = torch.meshgrid(torch.arange(depth_map.shape[0], device=depth_map.device, dtype=torch.float32),
                            torch.arange(depth_map.shape[1], device=depth_map.device, dtype=torch.float32), indexing="ij")
    z = depth_map / depth_scale
    return torch.stack([(ww - cx) * z / fx, (hh - cy) * z / fy, z], -1)


def depth2normal_geo(depth, k=31):
    """tensor(b,3,h,w) point map -> tensor(b,3,h,w) least-squares normals (not normalised)."""
    return torch.stack([_NormalFromXYZ.apply(depth[b].contiguous(), int(k)) for b in range(depth.shape[0])], 0)
