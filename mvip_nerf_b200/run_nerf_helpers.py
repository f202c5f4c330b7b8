"""Drop-in for the hot-path names of the reference's DS_NeRF/run_nerf_helpers.py.

Same names, argument meaning and return structures as the reference (citations per function); the
bodies call the sm_100a kernels of libmvip_nerf.so through `ops`.  Everything here needs CUDA tensors:
there is no CPU or eager-PyTorch fallback.

Not provided (out of scope, SURVEY.md §2 rows 7/8): NeRF_RGB, raw2outputs_with_normal, sample_sigma,
visualize_sigma, the tcnn model.
"""
import numpy as np
import torch
import torch.nn as nn

from . import ops

# Misc (run_nerf_helpers.py:15-18) — host-side lambdas, kept for callers that import them from here
img2mse = lambda x, y: torch.mean((x - y) ** 2)  # noqa: E731
img2l1 = lambda x, y: torch.mean(torch.abs(x - y))  # noqa: E731
mse2psnr = lambda x: -10. * torch.log(x) / torch.log(torch.tensor([10.], device=x.device))  # noqa: E731
to8b = lambda x: (255 * np.clip(x, 0, 1)).astype(np.uint8)  # noqa: E731


# ------------------------------------------------------------------------------------------------
# Positional encoding (run_nerf_helpers.py:22-70)
# ------------------------------------------------------------------------------------------------
class Embedder:
    """Same constructor kwargs and attributes (`embed`, `out_dim`, `kwargs`) as the reference class.
    Only the configuration get_embedder() builds is implemented by the kernel: include_input,
    log-sampled power-of-two bands, periodic_fns = [sin, cos]."""

    def __init__(self, **kwargs):
        self.kwargs = kwargs
        self.create_embedding_fn()

    def create_embedding_fn(self):
        kw = self.kwargs
        d = kw["input_dims"]
        n_freqs = kw["num_freqs"]
        fns = list(kw.get("periodic_fns", [torch.sin, torch.cos]))
        supported = (kw.get("include_input", True) and kw.get("log_sampling", True) and
                     kw["max_freq_log2"] == n_freqs - 1 and fns == [torch.sin, torch.cos])
        if not supported:
            raise NotImplementedError("Embedder: only include_input + log_sampling + [sin, cos] with "
                                      "max_freq_log2 == num_freqs-1 is implemented by the sm_100a kernels")
        self.input_dims = d
        self.num_freqs = n_freqs
        self.out_dim = d * (1 + 2 * n_freqs)

    def embed(self, inputs):
        return ops.embed(inputs, self.num_freqs)


class _EmbedFn:
    """Callable returned by get_embedder; carries `multires` so run_network can fuse it into the MLP kernel."""

    def __init__(self, embedder, multires):
        self.embedder = embedder
        self.multires = multires

    def __call__(self, x):
        return self.embedder.embed(x)


def get_embedder(multires, i=0):
    """(run_nerf_helpers.py:55-70) -> (embed callable, out_dim)"""
    if i == -1:
        return nn.Identity(), 3
    eo = Embedder(include_input=True, input_dims=3, max_freq_log2=multires - 1, num_freqs=multires,
                  log_sampling=True, periodic_fns=[torch.sin, torch.cos])
    return _EmbedFn(eo, multires), eo.out_dim


# ------------------------------------------------------------------------------------------------
# NeRF MLP (run_nerf_helpers.py:74-156)
# ------------------------------------------------------------------------------------------------
class _MLPFunction(torch.autograd.Function):
    """raw = NeRF(PE(pts), PE(dirs)).  backward gives the parameter gradients and, when the rays / points require grad, their
    gradient as well (mlp_input_grad, from the dZ images of the same backward): rays mode -> d ray batch (o, d, viewdir
    columns), points mode -> d pts, d dirs.  z_vals get none: the fine depths are detached in the reference (run.py:1812)."""

    @staticmethod
    def forward(ctx, net, mode, a, b, viewdir_offset, need_grad, *params):
        # need_grad is decided by the caller: grad mode is always off inside Function.forward
        packed = net.packed()
        kw = dict(rays=a, z_vals=b, viewdir_offset=viewdir_offset) if mode == "rays" else dict(pts=a, dirs=b)
        if need_grad:
            raw, stash = ops.mlp_forward(packed, want_stash=True, **kw)
            ctx.stash = stash
            ctx.packed = packed
            ctx.net, ctx.pack_gen = net, net._pack_gen
            ctx.mode, ctx.viewdir_offset = mode, viewdir_offset
            if ctx.needs_input_grad[2] or ctx.needs_input_grad[3]:
                ctx.save_for_backward(a, b)   # version-checked: an in-place change before backward raises
        else:
            raw = ops.mlp_forward(packed, **kw)
        ctx.need_grad = need_grad
        ctx.n_params = len(params)
        ctx.set_materialize_grads(False)
        return raw

    @staticmethod
    def backward(ctx, d_raw):
        if not ctx.need_grad or d_raw is None:
            return (None,) * (6 + ctx.n_params)
        if ctx.net._pack_gen != ctx.pack_gen:
            # the bf16 blob is shared and re-packed in place: dgrad would silently use the NEW weights (stock torch raises
            # its version-counter error in the same situation)
            raise RuntimeError("NeRF weights were re-packed (optimizer step / load_state_dict / invalidate_packed) between "
                               "this forward and its backward; run backward before changing the parameters")
        want_a, want_b = ctx.needs_input_grad[2], ctx.needs_input_grad[3] and ctx.mode == "points"
        grads, ws = ops.mlp_backward(ctx.packed, d_raw.contiguous(), ctx.stash, want_workspace=True)
        ctx.stash = None
        da = db = None
        if want_a or want_b:
            a, b = ctx.saved_tensors
            if ctx.mode == "rays":
                da = ops.mlp_input_grad(ctx.packed, ws, rays=a, z_vals=b, viewdir_offset=ctx.viewdir_offset)
            else:
                da, db = ops.mlp_input_grad(ctx.packed, ws, pts=a, dirs=b)
        return (None, None, da if want_a else None, db if want_b else None, None, None) + tuple(grads)


class NeRF(nn.Module):
    """Same constructor, parameter names and shapes as the reference module, so state_dicts interchange
    (pts_linears.{0..7}, views_linears.0, feature_linear, alpha_linear, rgb_linear).  forward(x[P,90]) takes
    the embedded input the reference's run_network builds; columns 0:3 and 63:66 of it are the raw point and
    view direction (include_input=True), which is what the fused kernel re-encodes on chip.

    The kernels implement the create_nerf configuration: D=8, W=256, input_ch=63, input_ch_views=27,
    skips=[4], use_viewdirs=True.  Anything else raises (no fallback)."""

    def __init__(self, D=8, W=256, input_ch=3, input_ch_views=3, output_ch=4, skips=[4], use_viewdirs=False):
        super().__init__()
        self.D, self.W = D, W
        self.input_ch, self.input_ch_views = input_ch, input_ch_views
        self.skips = list(skips)
        self.use_viewdirs = use_viewdirs
        if not (D == 8 and W == 256 and input_ch == 63 and input_ch_views == 27 and self.skips == [4] and use_viewdirs):
            raise NotImplementedError(
                "mvip_nerf_b200.NeRF implements D=8, W=256, input_ch=63, input_ch_views=27, skips=[4], "
                "use_viewdirs=True (create_nerf defaults, run.py:1487-1489); got D=%s W=%s input_ch=%s "
                "input_ch_views=%s skips=%s use_viewdirs=%s" % (D, W, input_ch, input_ch_views, skips, use_viewdirs))
        self.pts_linears = nn.ModuleList(
            [nn.Linear(input_ch, W)] +
            [nn.Linear(W, W) if i not in self.skips else nn.Linear(W + input_ch, W) for i in range(D - 1)])
        self.views_linears = nn.ModuleList([nn.Linear(input_ch_views + W, W // 2)])
        self.feature_linear = nn.Linear(W, W)
        self.alpha_linear = nn.Linear(W, 1)
        self.rgb_linear = nn.Linear(W // 2, 3)
        self._packed = None
        self._packed_key = None
        self._pack_gen = 0          # bumped by every re-pack; _MLPFunction checks it between forward and backward

    # -- packed bf16 weights ------------------------------------------------------------------------------------
    # The kernels read a bf16 operand blob, rebuilt lazily whenever a parameter is SEEN to have changed: torch's version
    # counters (optimizer.step, load_state_dict, p.copy_, .to()) or FusedAdam's epoch.  Writes that bypass both —
    # `p.data.copy_(w)`, `lin.weight.data = ...` keeping the same storage, raw-pointer writers — are invisible: call
    # invalidate_packed() after them.
    def _ordered_params(self):
        sd = dict(self.named_parameters())
        return [sd[n] for n in ops.PARAM_ORDER]

    def _pack_key(self, params):
        return (ops.param_epoch,) + tuple((p.data_ptr(), p._version) for p in params)

    def packed(self):
        params = self._ordered_params()
        key = self._pack_key(params)
        if self._packed is None or key != self._packed_key:
            self.repack(params)
        return self._packed

    def repack(self, params=None):
        """Rebuilds the bf16 blob from the current parameter values now (one launch, in place: CUDA-graph safe)."""
        params = self._ordered_params() if params is None else params
        self._packed = ops.mlp_pack(params, out=self._packed)
        self._packed_key = self._pack_key(params)
        self._pack_gen += 1
        return self._packed

    def invalidate_packed(self):
        """Call after writing parameters behind torch's back (`.data.copy_`, EMA / weight surgery through raw pointers)."""
        self._packed_key = None

    def _need_grad(self, params, *inputs):
        """stash for backward when the parameters OR the inputs (rays / points) require grad: a frozen network still
        back-propagates to its inputs (the full fused backward runs; its parameter gradients are dropped by autograd)"""
        return torch.is_grad_enabled() and (any(p.requires_grad for p in params) or any(t.requires_grad for t in inputs))

    def query_rays(self, ray_batch, z_vals):
        """raw [N,S,4] for pts = o + d*z of every (ray, sample); viewdir = last 3 columns of ray_batch."""
        params = self._ordered_params()
        raw = _MLPFunction.apply(self, "rays", ray_batch, z_vals, ray_batch.shape[1] - 3, self._need_grad(params, ray_batch),
                                 *params)
        return raw.view(z_vals.shape[0], z_vals.shape[1], 4)

    def query_points(self, pts, dirs):
        """raw [P,4] for explicit points / directions ([P,3] each, any row stride); differentiable w.r.t. pts and dirs."""
        params = self._ordered_params()
        return _MLPFunction.apply(self, "points", pts, dirs, 0, self._need_grad(params, pts, dirs), *params)

    def forward(self, x):
        """Gradients reach the parameters only, not x: the kernel re-encodes columns 0:3 and 63:66 of x, so the reference's
        gradient for the other 84 (embedded) columns has no counterpart.  Use query_points for d pts / d dirs."""
        if x.shape[-1] != self.input_ch + self.input_ch_views:
            raise RuntimeError("NeRF.forward expects [..., %d] embedded inputs" % (self.input_ch + self.input_ch_views))
        flat = x.reshape(-1, x.shape[-1])
        out = self.query_points(flat[:, 0:3].detach(), flat[:, self.input_ch:self.input_ch + 3].detach())
        return out.reshape(*x.shape[:-1], 4)

    def load_weights_from_keras(self, weights):
        """(run_nerf_helpers.py:129-156) same index convention as the reference."""
        assert self.use_viewdirs, "Not implemented if use_viewdirs=False"
        dev = self.feature_linear.weight.device

        def put(lin, iw):
            lin.weight.data = torch.from_numpy(np.transpose(weights[iw])).to(dev)
            lin.bias.data = torch.from_numpy(np.transpose(weights[iw + 1])).to(dev)
        for i in range(self.D):
            put(self.pts_linears[i], 2 * i)
        put(self.feature_linear, 2 * self.D)
        put(self.views_linears[0], 2 * self.D + 2)
        put(self.rgb_linear, 2 * self.D + 4)
        put(self.alpha_linear, 2 * self.D + 6)
        self.invalidate_packed()


# ------------------------------------------------------------------------------------------------
# Ray helpers (run_nerf_helpers.py:249-300) under the reference's names, as torch ops on whatever device the pose is on
# (callers such as the training loop's ray precomputation, run.py:620, :869, use them directly).  render() itself does not
# call them: it gets the whole [N, 8|11] ray batch from ONE kernel (ops.rays_from_pose / ops.rays_pack, csrc/rays.cu),
# bit-exact against these formulas evaluated by torch on the CPU.
# ------------------------------------------------------------------------------------------------
def get_rays(H, W, focal, c2w):
    dev = c2w.device if torch.is_tensor(c2w) else None
    c2w = torch.as_tensor(c2w, dtype=torch.float32, device=dev)
    xs = torch.linspace(0, W - 1, W, device=c2w.device)
    ys = torch.linspace(0, H - 1, H, device=c2w.device)
    j, i = torch.meshgrid(ys, xs, indexing="ij")          # i: column index, j: row index, both [H,W]
    dirs = torch.stack([(i - W * .5) / focal, -(j - H * .5) / focal, -torch.ones_like(i)], -1)
    rays_d = torch.sum(dirs[..., None, :] * c2w[:3, :3], -1)
    rays_o = c2w[:3, -1].expand(rays_d.shape)
    return rays_o, rays_d


def get_rays_np(H, W, focal, c2w):
    i, j = np.meshgrid(np.arange(W, dtype=np.float32), np.arange(H, dtype=np.float32), indexing="xy")
    dirs = np.stack([(i - W * .5) / focal, -(j - H * .5) / focal, -np.ones_like(i)], -1)
    rays_d = np.sum(dirs[..., np.newaxis, :] * c2w[:3, :3], -1)
    rays_o = np.broadcast_to(c2w[:3, -1], np.shape(rays_d))
    return rays_o, rays_d


def ndc_rays(H, W, focal, near, rays_o, rays_d):
    t = -(near + rays_o[..., 2]) / rays_d[..., 2]
    rays_o = rays_o + t[..., None] * rays_d
    sx, sy = -1. / (W / (2. * focal)), -1. / (H / (2. * focal))
    o = torch.stack([sx * rays_o[..., 0] / rays_o[..., 2], sy * rays_o[..., 1] / rays_o[..., 2],
                     1. + 2. * near / rays_o[..., 2]], -1)
    d = torch.stack([sx * (rays_d[..., 0] / rays_d[..., 2] - rays_o[..., 0] / rays_o[..., 2]),
                     sy * (rays_d[..., 1] / rays_d[..., 2] - rays_o[..., 1] / rays_o[..., 2]),
                     -2. * near / rays_o[..., 2]], -1)
    return o, d


# ------------------------------------------------------------------------------------------------
# Hierarchical sampling (run_nerf_helpers.py:304-347)
# ------------------------------------------------------------------------------------------------
def sample_pdf(bins, weights, N_samples, det=False, pytest=False, return_inds=False):
    """-> samples [N, N_samples].  u is drawn on the host exactly where the reference draws it: det ->
    torch.linspace row; otherwise torch.rand; pytest -> numpy's seeded stream (helpers:318-327).
    The result carries no gradient (its only caller detaches it, run.py:1812)."""
    dev = bins.device
    lead = bins.shape[:-1]
    bins2 = bins.detach().reshape(-1, bins.shape[-1])
    w2 = weights.detach().reshape(-1, weights.shape[-1])
    n = bins2.shape[0]
    if det:
        u = torch.linspace(0., 1., steps=N_samples, device=dev)
    else:
        u = torch.rand([n, N_samples], device=dev)
    if pytest:
        np.random.seed(0)
        if det:
            u = torch.Tensor(np.linspace(0., 1., N_samples)).to(dev)
        else:
            u = torch.Tensor(np.random.rand(n, N_samples)).to(dev)
    samples, inds, _ = ops.sample_pdf(bins2, w2, u, want_inds=return_inds)
    samples = samples.reshape(*lead, N_samples)
    if return_inds:
        return samples, inds.reshape(*lead, N_samples)
    return samples


# ------------------------------------------------------------------------------------------------
# Alpha compositing (run_nerf_helpers.py:350-404)
# ------------------------------------------------------------------------------------------------
class _CompositeFunction(torch.autograd.Function):
    """raw2outputs as one forward and one backward kernel.  With `target_rgb` / `target_disp` the photometric losses are fused in
    (img2mse of rgb / rgb0 / disp as train() uses it, run.py:1000-1027): a seventh output sq [2] = (sum (rgb_map - target_rgb)^2,
    sum (disp_map - target_disp)^2), whose gradient is applied inside the backward kernel from the recomputed maps."""

    @staticmethod
    def forward(ctx, raw, z_vals, rays_d, noise, white_bkgd, need_alpha, detach_weights, target_rgb=None, target_disp=None):
        fused = target_rgb is not None or target_disp is not None
        outs = ops.composite_forward(raw, z_vals, rays_d, noise, white_bkgd, need_alpha, target_rgb, target_disp)
        rgb, disp, acc, weights, depth, alpha = outs[:6]
        ctx.set_materialize_grads(False)   # unused outputs arrive as None (the kernel takes NULL = zeros): no fill kernels
        ctx.save_for_backward(raw, z_vals, rays_d, noise, target_rgb, target_disp)
        ctx.flags = (bool(white_bkgd), bool(detach_weights), bool(need_alpha))
        if not need_alpha:
            alpha = raw.new_empty(0)
            ctx.mark_non_differentiable(alpha)
        sq = outs[6] if fused else raw.new_empty(0)
        if not fused:
            ctx.mark_non_differentiable(sq)
        return rgb, disp, acc, weights, depth, alpha, sq

    @staticmethod
    def backward(ctx, g_rgb, g_disp, g_acc, g_weights, g_depth, g_alpha, g_sq):
        raw, z_vals, rays_d, noise, target_rgb, target_disp = ctx.saved_tensors
        white, detach_w, need_alpha = ctx.flags
        if all(g is None for g in (g_rgb, g_disp, g_acc, g_weights, g_depth, g_alpha, g_sq)):
            return (None,) * 9
        want_d = ctx.needs_input_grad[2]
        out = ops.composite_backward(raw, z_vals, rays_d, noise, white, detach_w, g_rgb, g_disp, g_acc, g_depth,
                                     g_weights, g_alpha if need_alpha else None, target_rgb, target_disp, g_sq, want_rays_d=want_d)
        d_raw, d_rays_d = out if want_d else (out, None)
        return (d_raw, None, d_rays_d) + (None,) * 6


def raw2outputs(raw, z_vals, rays_d, raw_noise_std=0, white_bkgd=False, pytest=False, need_alpha=False,
                detach_weights=False, _noise=None, _mse=None):
    """-> (rgb_map, disp_map, acc_map, weights, depth_map, alpha|None), differentiable w.r.t. raw and rays_d (through
    dists * |rays_d|); z_vals get no gradient.
    `_mse=(target_rgb | None, target_disp | None)` (ours): the squared-error sums of img2mse come out of the same kernels as a
    seventh element sq [2]."""
    noise = _noise
    if noise is None and raw_noise_std > 0.:
        noise = torch.randn(raw[..., 3].shape, device=raw.device) * raw_noise_std
        if pytest:   # the reference overwrites with UNIFORM numpy randoms here (helpers:377-381)
            np.random.seed(0)
            noise = torch.Tensor(np.random.rand(*list(raw[..., 3].shape)) * raw_noise_std).to(raw.device)
    t_rgb, t_disp = _mse if _mse is not None else (None, None)
    rgb, disp, acc, weights, depth, alpha, sq = _CompositeFunction.apply(raw, z_vals, rays_d, noise, white_bkgd, need_alpha,
                                                                         detach_weights, t_rgb, t_disp)
    if _mse is not None:
        return rgb, disp, acc, weights, depth, (alpha if need_alpha else None), sq
    return rgb, disp, acc, weights, depth, (alpha if need_alpha else None)


# ------------------------------------------------------------------------------------------------
# Depth -> normal map (run.py:1909-1940); exported from run.py under the reference's names as well
# ------------------------------------------------------------------------------------------------
class _NormalFromDepth(torch.autograd.Function):
    @staticmethod
    def forward(ctx, depth, fx, fy, cx, cy, k):
        ctx.save_for_backward(depth)
        ctx.cam = (fx, fy, cx, cy, k)
        return ops.normal_forward(depth, fx, fy, cx, cy, k)

    @staticmethod
    def backward(ctx, g):
        (depth,) = ctx.saved_tensors
        fx, fy, cx, cy, k = ctx.cam
        return ops.normal_backward(depth, fx, fy, cx, cy, g, k), None, None, None, None, None


class _NormalFromXYZ(torch.autograd.Function):
    @staticmethod
    def forward(ctx, xyz, k):
        ctx.save_for_backward(xyz)
        ctx.k = k
        return ops.normal_forward_xyz(xyz, k)

    @staticmethod
    def backward(ctx, g):
        (xyz,) = ctx.saved_tensors
        return ops.normal_backward_xyz(xyz, g, ctx.k), None


def depth2normal(depth, depth_cam_matrix, k=31):
    """Fused depth [h,w] -> normal [1,3,h,w] (== depth2normal_geo(depth2xyz_torch(depth, K)...), run.py:960-964)."""
    K = depth_cam_matrix
    n = _NormalFromDepth.apply(depth, float(K[0][0]), float(K[1][1]), float(K[0][2]), float(K[1][2]), int(k))
    return n.unsqueeze(0)
