"""Multi-GPU plumbing: one process per GPU (torchrun), rays sharded across ranks.

Replaces the reference's nn.DataParallel (run.py:1491,1527), which re-broadcasts the weights and
scatters/gathers [P,90] inputs on every MLP call.  Here the weights are replicated once, each rank
renders its contiguous slice of the ray batch with no data-path communication, and

  * a render ends with ONE gather of (rgb, disp, acc, depth) = 24 B/ray to rank 0;
  * a training step ends with ONE sum-allreduce of the flattened fp32 parameter gradients of BOTH networks
    (2 x 595,844 x 4 B = 4.77 MB; `GraphedTrainStep` carves the two flat buffers from one arena) over NCCL/NVLink, issued
    after the backward pass — also inside the step's captured CUDA graph.  allreduce_grads() is the eager form (one call
    per network).  GradSync(overlap=True) CAN start a network's bucket from a post-accumulate-grad hook the moment its 24
    gradients exist (the fine branch finishes first; the branches are independent: z_samples is detached, run.py:1812),
    but it is NOT the default: the fused MLP backward is a persistent kernel that needs every SM, and an NCCL kernel
    scheduled next to it only delays its CTAs (measured on 2 B200: 3.74 - 3.83 ms per step overlapped, 3.64 ms with one
    bucket after the backward; DESIGN.md section 6).

The host logic is backend-agnostic (gloo on CPU tensors in tests/, nccl on the GPU box).
"""
import os

import torch
import torch.distributed as dist


def init_from_env(backend=None):
    """Reads RANK / LOCAL_RANK / WORLD_SIZE / MASTER_* (torchrun).  Returns (rank, world, local_rank)."""
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1 and not dist.is_initialized():
        if backend is None:
            backend = "nccl" if torch.cuda.is_available() else "gloo"
        if backend == "nccl":
            torch.cuda.set_device(local)
        dist.init_process_group(backend=backend, rank=rank, world_size=world)
    elif torch.cuda.is_available():
        torch.cuda.set_device(local)
    return rank, world, local


def world():
    return dist.get_world_size() if dist.is_initialized() else 1


def rank():
    return dist.get_rank() if dist.is_initialized() else 0


def shard_bounds(n, r=None, w=None):
    """Contiguous, balanced slice [lo, hi) of n units for rank r of w (first n % w ranks get one extra)."""
    r = rank() if r is None else r
    w = world() if w is None else w
    base, extra = divmod(n, w)
    lo = r * base + min(r, extra)
    return lo, lo + base + (1 if r < extra else 0)


def shard_rows(t, r=None, w=None):
    lo, hi = shard_bounds(t.shape[0], r, w)
    return t[lo:hi]


def gather_rows(local, n_total, dst=0):
    """Concatenates per-rank row slices (shard_bounds order) on rank dst; other ranks get None.
    One collective: all ranks pad to the largest shard and all_gather into a single buffer."""
    if world() == 1:
        return local
    w = world()
    return _gather_uneven(local, [hi - lo for lo, hi in (shard_bounds(n_total, r, w) for r in range(w))], dst)


def render_sharded(render_fn, rays_flat, **kwargs):
    """Renders rank-local rows of rays_flat [N, C] with render_fn(rows, **kwargs) -> dict of [n, ...] tensors and
    gathers rgb_map / disp_map / acc_map / depth_map on rank 0 as one packed [N, 6] tensor (24 B/ray)."""
    n = rays_flat.shape[0]
    ret = render_fn(shard_rows(rays_flat), **kwargs)
    packed = torch.cat([ret["rgb_map"], ret["disp_map"][:, None], ret["acc_map"][:, None], ret["depth_map"][:, None]], -1)
    full = gather_rows(packed.contiguous(), n)
    if full is None:
        return None
    return {"rgb_map": full[:, 0:3], "disp_map": full[:, 3], "acc_map": full[:, 4], "depth_map": full[:, 5]}


def view_row_bands(n_views, H, r=None, w=None):
    """Rows of a stack of n_views images of H rows, split evenly over the ranks: rank r gets the contiguous range
    shard_bounds(n_views * H) of the global row index; returned as [(view, first_row, n_rows)] (a range may straddle views)."""
    lo, hi = shard_bounds(n_views * H, r, w)
    bands = []
    while lo < hi:
        v, i0 = divmod(lo, H)
        n = min(H - i0, hi - lo)
        bands.append((v, i0, n))
        lo += n
    return bands


def render_views_sharded(render_fn, poses, H, W, focal, near, far, normal_k=31, with_normals=True, **kwargs):
    """The guidance render batch (BASELINE cfg 5; render_path_4view + the normal-map branch of train(), DS_NeRF/run.py:948-982):
    V views of H x W, rgb + disp + acc + depth per pixel and, on rank 0, the depth-derived normal map of each view.

    Rows of the V*H image rows are sharded over the ranks (row bands -> mvip_rays_from_pose windows), every rank renders its
    bands with render_fn(H, W, focal, c2w=pose, patch=(i0, 0, n, W), near=, far=, **kwargs) -> [rgb, disp, acc, depth, extras],
    ONE gather of 24 B/pixel brings them to rank 0, which runs the normal-map kernels (a 31 x 31 stencil over the whole
    image; 24 B/pixel of traffic).  Returns on rank 0 a dict of [V,H,W,...] tensors (+ 'normal' [V,3,H,W], mapped to
    (n + 1) / 2 as in run.py:965); None on the other ranks.  No pose gradients: the gathered images are leaves."""
    from .run_nerf_helpers import depth2normal
    V = len(poses)
    kwargs = {k: v for k, v in kwargs.items() if k not in ("near", "far")}     # bounds merged into the kwargs (run.py:554-559)
    pieces = []
    for v, i0, n in view_row_bands(V, H):
        rgb, disp, acc, depth, _ = render_fn(H, W, focal, c2w=poses[v][:3, :4], patch=(i0, 0, n, W), near=near, far=far, **kwargs)
        pieces.append(torch.cat([rgb.reshape(-1, 3), disp.reshape(-1, 1), acc.reshape(-1, 1), depth.reshape(-1, 1)], -1))
    some = poses[0]
    dev = some.device if torch.is_tensor(some) and some.is_cuda else (
        torch.device("cuda", torch.cuda.current_device()) if torch.cuda.is_available() else torch.device("cpu"))
    packed = torch.cat(pieces, 0) if pieces else torch.empty((0, 6), device=dev)
    # row bands are whole rows, so the row-sharded gather of pixels == gather_rows with W pixels per row
    full = _gather_uneven(packed.contiguous(), [(b[1] - b[0]) * W for b in (shard_bounds(V * H, r, world()) for r in range(world()))])
    if full is None:
        return None
    full = full.view(V, H, W, 6)
    out = {"rgb_map": full[..., 0:3], "disp_map": full[..., 3], "acc_map": full[..., 4], "depth_map": full[..., 5]}
    if with_normals:
        K = [[focal, 0., W / 2], [0., focal, H / 2], [0., 0., 1.]]
        out["normal"] = torch.cat([(depth2normal(out["depth_map"][v].contiguous(), K, normal_k) + 1) / 2 for v in range(V)], 0)
    return out


def _gather_uneven(local, sizes, dst=0):
    """all ranks contribute `sizes[r]` rows; rank dst gets the concatenation (one padded all_gather), others None."""
    if world() == 1:
        return local
    w = world()
    max_rows = max(sizes)
    pad = local.new_zeros((max_rows,) + tuple(local.shape[1:]))
    pad[:local.shape[0]] = local
    out = local.new_empty((w * max_rows,) + tuple(local.shape[1:]))
    if local.is_cuda:
        dist.all_gather_into_tensor(out, pad)
    else:
        dist.all_gather([out[r * max_rows:(r + 1) * max_rows] for r in range(w)], pad)
    if rank() != dst:
        return None
    return torch.cat([out[r * max_rows:r * max_rows + sizes[r]] for r in range(w)], 0)


def _scatter_uneven(full, sizes, like, src=0):
    """inverse of _gather_uneven: rank src holds `full` [sum(sizes), ...]; every rank gets its rows (one padded scatter)."""
    if world() == 1:
        return full
    w = world()
    max_rows = max(sizes)
    out = like.new_empty((max_rows,) + tuple(like.shape[1:]))
    chunks = None
    if rank() == src:
        chunks, off = [], 0
        for n in sizes:
            c = like.new_zeros((max_rows,) + tuple(like.shape[1:]))
            c[:n] = full[off:off + n]
            chunks.append(c)
            off += n
    dist.scatter(out, chunks, src=src)
    return out[:sizes[rank()]]


class ShardedGuidanceViews:
    """Guidance views WITH gradients across the GPUs of one box (BASELINE cfg 5 in its training role: the collaborative /
    normal-map branches of train(), DS_NeRF/run.py:948-984, render their views with autograd on).

        g = ShardedGuidanceViews(render_kwargs, poses, H, W, focal, near, far)
        out = g.forward()            # all ranks; rank 0 gets {'rgb_map' [V,H,W,3], 'disp_map', 'acc_map', 'depth_map'} as
                                     # gradient-carrying leaves (+ 'normal' [V,3,H,W] built from depth_map with autograd), others None
        loss(out).backward()         # rank 0 only: stock-PyTorch guidance loss (SDS, ...) on the gathered images
        g.backward()                 # all ranks: image gradients scattered back (24 B/ray), every rank back-propagates ITS rows
                                     # with deferred re-rendering (run._DeferredRays), then one gradient allreduce per network

    Communication: one gather (24 B/ray), one scatter (24 B/ray), one 4.77 MB allreduce.  Every rank ends with the full
    parameter gradient in .grad, exactly as after dist.allreduce_grads in the ray-batch step.  Gradients reach the network
    parameters only, not the poses: each rank would hold the pose gradient of its own rows, and nothing reduces those."""

    def __init__(self, render_kwargs, poses, H, W, focal, near, far, chunk=8192, with_normals=True, normal_k=31):
        from . import run as mrun
        self.run = mrun
        self.kw = dict(render_kwargs)
        self.poses, self.H, self.W, self.focal, self.near, self.far = poses, int(H), int(W), focal, near, far
        self.chunk, self.with_normals, self.normal_k = int(chunk), with_normals, normal_k
        self.nets = mrun._net_params(self.kw)
        self.outs = self.leaf = None

    def _sizes(self):
        V = len(self.poses)
        return [(b[1] - b[0]) * self.W for b in (shard_bounds(V * self.H, r, world()) for r in range(world()))]

    def forward(self):
        from . import ops
        from .run_nerf_helpers import depth2normal
        V, H, W = len(self.poses), self.H, self.W
        use_viewdirs = self.kw.get("use_viewdirs", False)
        ndc = self.kw.get("ndc", True)
        pieces = [ops.rays_from_pose(H, W, self.focal, self.poses[v][:3, :4], self.near, self.far, use_viewdirs=use_viewdirs,
                                     patch=(i0, 0, n, W), ndc=ndc) for v, i0, n in view_row_bands(V, H)]
        kw = {k: v for k, v in self.kw.items() if k not in ("ndc", "use_viewdirs", "near", "far")}
        params = [p for _, ps in self.nets for p in ps]
        if pieces:
            rays = torch.cat(pieces, 0) if len(pieces) > 1 else pieces[0]
            holder = {}
            outs = self.run._DeferredRays.apply(rays, self.chunk, kw, holder, *params)
            ret = dict(zip(holder["keys"], outs))
            self.outs = [ret["rgb_map"], ret["disp_map"], ret["acc_map"], ret["depth_map"]]
            packed = torch.cat([self.outs[0].detach(), self.outs[1].detach()[:, None], self.outs[2].detach()[:, None],
                                self.outs[3].detach()[:, None]], -1)
        else:       # more ranks than image rows
            self.outs = None
            packed = params[0].new_empty((0, 6))
        full = _gather_uneven(packed.contiguous(), self._sizes())
        if full is None:
            return None
        self.leaf = full.detach().requires_grad_(True)
        img = self.leaf.view(V, H, W, 6)
        out = {"rgb_map": img[..., 0:3], "disp_map": img[..., 3], "acc_map": img[..., 4], "depth_map": img[..., 5]}
        if self.with_normals:
            K = [[self.focal, 0., W / 2], [0., self.focal, H / 2], [0., 0., 1.]]
            out["normal"] = torch.cat([(depth2normal(out["depth_map"][v].contiguous(), K, self.normal_k) + 1) / 2 for v in range(V)], 0)
        return out

    def backward(self):
        sizes = self._sizes()
        like = self.outs[0].new_empty((0, 6)) if self.outs is not None else self.nets[0][1][0].new_empty((0, 6))
        g_full = None
        if rank() == 0:
            g_full = self.leaf.grad if self.leaf.grad is not None else torch.zeros_like(self.leaf)
        g = _scatter_uneven(g_full, sizes, like)
        if self.outs is not None and g.shape[0] > 0:
            torch.autograd.backward(self.outs, [g[:, 0:3].contiguous(), g[:, 3].contiguous(), g[:, 4].contiguous(),
                                                g[:, 5].contiguous()])
        for _, ps in self.nets:        # ranks whose rows carried no gradient still take part in the collective
            for p in ps:
                if p.grad is None:
                    p.grad = torch.zeros_like(p)
        allreduce_grads([ps for _, ps in reversed(self.nets)])
        self.outs = self.leaf = None


def _flat_view(grads):
    """If the gradient tensors are consecutive views of ONE contiguous buffer (what ops.mlp_backward returns: 24 views of
    one flat fp32 tensor per network), returns that buffer as a 1-D tensor sharing their memory; otherwise None."""
    g0 = grads[0]
    if not g0.is_contiguous():
        return None
    st = g0.untyped_storage()
    off = g0.storage_offset()
    total = 0
    for g in grads:
        if (g.dtype != g0.dtype or g.device != g0.device or not g.is_contiguous() or
                g.untyped_storage().data_ptr() != st.data_ptr() or g.storage_offset() != off + total):
            return None
        total += g.numel()
    return torch.empty(0, dtype=g0.dtype, device=g0.device).set_(st, off, (total,))


class GradAllReducer:
    """Sum-allreduce of the gradients of a list of parameters as ONE flat fp32 bucket (async).  When the gradients already
    live back to back in one buffer (the MLP backward writes them that way) the collective runs IN PLACE on it: no
    concatenation before and no 24 copy kernels after."""

    def __init__(self, params):
        self.params = [p for p in params]
        self.handle = None
        self.flat = None
        self.in_place = False

    def start(self):
        if world() == 1:
            return
        grads = [p.grad if p.grad is not None else torch.zeros_like(p) for p in self.params]
        view = _flat_view(grads) if all(p.grad is not None for p in self.params) else None
        self.in_place = view is not None
        self.flat = view if self.in_place else torch.cat([g.reshape(-1) for g in grads])
        self.handle = dist.all_reduce(self.flat, op=dist.ReduceOp.SUM, async_op=True)

    def start_if_contiguous(self):
        """Starts the collective only if it can run in place on one contiguous buffer; -> whether it did."""
        if world() == 1 or any(p.grad is None for p in self.params):
            return False
        view = _flat_view([p.grad for p in self.params])
        if view is None:
            return False
        self.in_place, self.flat = True, view
        self.handle = dist.all_reduce(self.flat, op=dist.ReduceOp.SUM, async_op=True)
        return True

    def finish(self):
        if self.handle is None:
            return
        self.handle.wait()
        if not self.in_place:
            off = 0
            for p in self.params:
                n = p.numel()
                g = self.flat[off:off + n].view_as(p)
                if p.grad is None:
                    p.grad = g.clone()
                else:
                    p.grad.copy_(g)
                off += n
        self.handle, self.flat = None, None


class GradSync:
    """Gradient allreduce, one bucket per network.  overlap=True: a bucket is started from post-accumulate-grad hooks as soon
    as ALL gradients of its network have been accumulated, i.e. while the rest of the backward pass still runs; finish() joins
    them (and starts the buckets of networks that received no gradient, so every rank issues the same collectives).
    overlap=False: finish() starts and joins all buckets after the backward pass.  The fused MLP backward is a persistent
    kernel that needs every SM (its CTA pairs wait for each other's tiles): an NCCL kernel that gets SMs first keeps part of its
    grid from becoming resident until the collective (and the peer it waits for) is done, so the graphed train step does not
    overlap (measured on 2 B200: 3.74 - 4.00 ms per step overlapped against 3.64 ms with one bucket after the backward).

        sync = GradSync([fine_params, coarse_params])
        loss.backward(); sync.finish(); optimizer.step()
    """

    def __init__(self, param_groups, overlap=True):
        self.overlap = bool(overlap)
        self.groups = [list(ps) for ps in param_groups]
        self.reducers = [GradAllReducer(ps) for ps in self.groups]
        self._all = GradAllReducer([p for ps in self.groups for p in ps])
        self.count = [0] * len(self.groups)
        self.started = [False] * len(self.groups)
        self.hooks = []
        for gi, ps in enumerate(self.groups):
            for p in ps:
                self.hooks.append(p.register_post_accumulate_grad_hook(lambda _p, gi=gi: self._on_grad(gi)))

    def _on_grad(self, gi):
        self.count[gi] += 1
        if self.count[gi] == len(self.groups[gi]):
            self.count[gi] = 0
            if world() > 1 and self.overlap and not self.started[gi]:
                self.reducers[gi].start()
                self.started[gi] = True

    def finish(self):
        if world() > 1:
            if not any(self.started) and self._all.start_if_contiguous():
                self._all.finish()          # the gradients of all networks are one contiguous range: ONE collective
            else:
                for gi, r in enumerate(self.reducers):
                    if not self.started[gi]:
                        r.start()
                for r in self.reducers:
                    r.finish()
        self.count = [0] * len(self.groups)
        self.started = [False] * len(self.groups)

    def remove(self):
        for h in self.hooks:
            h.remove()
        self.hooks = []


def allreduce_grads(param_groups):
    """param_groups: iterable of parameter lists (e.g. [coarse params, fine params]); one bucket each."""
    reducers = [GradAllReducer(ps) for ps in param_groups]
    for r in reducers:
        r.start()
    for r in reducers:
        r.finish()
