"""One training step as CUDA graphs (B200: launch-bound glue replaced by graph replays).

A cfg-2 step is ~45 kernel launches, 16 of them ours; the three MLP kernels take 90 % of the GPU time and everything else
(random draws, the loss and its autograd, ray packing, sampling, compositing, Adam, the bf16 re-pack) is a string of
5-20 us kernels whose launch gaps — and, end to end, the Python that issues them after every `loss.item()` — add up to
~10 % of the step.  GraphedTrainStep captures

    rays -> render() -> loss -> backward      (fresh random draws on every replay: torch registers the CUDA generator with
                                               the graph and advances its offset)
         -> gradient allreduce (N > 1)        ONE NCCL bucket for both networks (their flat gradient buffers are carved from
                                               one arena), issued after the backward: the fused backward owns every SM, an
                                               overlapped collective only delays its CTAs (dist.GradSync(overlap=True) exists
                                               and measured slower, DESIGN.md section 6)
         -> Adam (lr and step number read from device memory) -> re-pack of the bf16 weight blobs

as ONE graph, once, after warm-up, and replays it.  With `poses=` (a cameras.CameraPoses table) the step also refines the camera
poses: `__call__(pixels, target)` copies (view, row, col) indices instead of rays, and the graph runs the pose module, the
pose-table ray kernel and its backward, and a second FusedAdam on the pose parameters (its own device lr / step).  (`nccl_in_graph=False` keeps the collectives out of the capture: graph A =
render + loss + backward, eager allreduce, graph B = Adam + re-pack.)  Inputs live in static buffers; `__call__(rays, target)` copies into them (from pinned
host memory for the end-to-end path) and returns the loss as a device scalar.  Same arithmetic as the eager step: the captured
launches ARE the eager step's launches.
"""
import torch

from . import dist as mdist
from . import ops, run
from .run_nerf_helpers import img2mse


def default_loss(rgb, disp, acc, depth, extras, target, scale):
    """img2mse(rgb, target) + img2mse(rgb0, target)   (run.py:1000, 1024-1026), scaled for data-parallel averaging.
    When the render was given `_mse=(target, None)` the squared-error sums come out of the compositing kernels (`sqerr`,
    `sqerr0`) and their gradient goes back into the compositing backward: the ~20 elementwise / reduction / autograd kernels
    of the two img2mse calls become three scalar ops."""
    if "sqerr" in extras:
        sq = extras["sqerr"][0]
        if "sqerr0" in extras:
            sq = sq + extras["sqerr0"][0]
        return sq * (scale / rgb.numel())
    loss = img2mse(rgb, target)
    if "rgb0" in extras:
        loss = loss + img2mse(extras["rgb0"], target)
    return loss * scale


def step_syncs(net_groups, pose_params, overlap=False):
    """The gradient collectives of one data-parallel step -> (networks' GradSync | None, pose table's GradSync | None).  The pose
    table is its own small bucket, finished after the networks' one.  Each rank holds the gradient of its own rays; finish() on
    both leaves the sums over the ranks."""
    return (mdist.GradSync(net_groups, overlap=overlap) if net_groups else None,
            mdist.GradSync([list(pose_params)], overlap=False) if pose_params else None)


class GraphedTrainStep:
    """One CUDA-graph replay per training step.

    Without `poses`, gradients reach the network parameters only: the ray batch is copied into the graph's static buffers, so
    rays or poses that require grad get no gradient here.  With `poses` (a cameras.CameraPoses) and `pose_optimizer` (a
    FusedAdam over poses.parameters()), each call takes pixels [n_rays, 3] = (view, row, col) and the step renders those pixels
    of the table's current poses, back-propagates to the networks and to the table, and updates both.  `optimizer` may then be
    None when every network parameter is frozen (pose estimation against a trained scene): the networks get no Adam and no
    re-pack."""

    def __init__(self, render_kwargs_train, optimizer, H, W, focal, n_rays, near=None, far=None, chunk=1024 * 32, loss_fn=default_loss,
                 target_shape=None, warmup=3, device=None, nccl_in_graph=True, overlap_allreduce=False, poses=None,
                 pose_optimizer=None):
        if not torch.cuda.is_available():
            raise RuntimeError("GraphedTrainStep needs a CUDA device (no CPU fallback)")
        if (poses is None) != (pose_optimizer is None):
            raise ValueError("GraphedTrainStep: poses and pose_optimizer go together")
        if optimizer is None and poses is None:
            raise ValueError("GraphedTrainStep: an optimizer is needed unless a pose table is refined")
        self.kw = dict(render_kwargs_train)
        # train() merges the scene bounds into the kwargs (run.py:554-559): accept both forms
        kw_near, kw_far = self.kw.pop("near", None), self.kw.pop("far", None)
        near = kw_near if near is None else near
        far = kw_far if far is None else far
        if near is None or far is None:
            raise ValueError("GraphedTrainStep: near / far must be given (as arguments or inside render_kwargs_train)")
        self.opt = optimizer
        self.dev = device or torch.device("cuda", torch.cuda.current_device())
        self.args = (H, W, focal)
        self.chunk, self.near, self.far = chunk, near, far
        self.loss_fn = loss_fn
        # the default photometric loss is fused into the compositing kernels (64 / 128 samples per ray: what those kernels cover)
        self.fused_loss = (loss_fn is default_loss and self.kw.get("N_samples") == 64 and self.kw.get("N_importance") in (0, 64)
                           and target_shape is None)
        self.scale = 1.0 / mdist.world()
        self.poses, self.pose_opt = poses, pose_optimizer
        if poses is None:
            self.rays = torch.zeros((2, n_rays, 3), device=self.dev)
        else:
            self.pixels = torch.zeros((n_rays, 3), device=self.dev, dtype=torch.int32)
        self.target = torch.zeros(tuple(target_shape or (n_rays, 3)), device=self.dev)
        if optimizer is None:
            if any(p.requires_grad for _, ps in run._net_params(self.kw) for p in ps):
                raise ValueError("GraphedTrainStep: optimizer=None needs every network parameter frozen (requires_grad=False)")
            self.nets, self.groups = [], []
        else:
            self.nets = [n for n, _ in run._net_params(self.kw)]
            self.groups = [ps for _, ps in reversed(run._net_params(self.kw))]      # fine first: its gradients exist first
        self.pose_params = [] if poses is None else list(poses.parameters())
        self.opts = [o for o in (optimizer, pose_optimizer) if o is not None]
        self.warmup = warmup
        self.graph_a = self.graph_b = None
        self.loss = None
        self.one_graph = bool(nccl_in_graph) or mdist.world() == 1
        self.sync, self.pose_sync = (step_syncs(self.groups, self.pose_params, overlap_allreduce)
                                     if (self.one_graph and mdist.world() > 1) else (None, None))
        n_grad = sum(p.numel() for ps in self.groups for p in ps)
        self.grad_arena = torch.empty(n_grad, device=self.dev, dtype=torch.float32) if (mdist.world() > 1 and n_grad) else None

    # -- the two halves of the step, exactly as the eager loop runs them -----------------------------------------------
    def _forward_backward(self):
        for opt in self.opts:
            opt.zero_grad(set_to_none=True)
        if self.grad_arena is not None:       # both networks' gradients back to back: one allreduce (dist.GradSync.finish)
            ops.grad_arena.begin(self.grad_arena)
        try:
            return self._forward_backward_body()
        finally:
            ops.grad_arena.end()

    def _forward_backward_body(self):
        H, W, focal = self.args
        mse = {"_mse": (self.target, None)} if self.fused_loss else {}
        src = {"rays": self.rays} if self.poses is None else {"c2w": self.poses(), "pixels": self.pixels}
        rgb, disp, acc, depth, extras = run.render(H, W, focal, chunk=self.chunk, near=self.near, far=self.far, **src, **mse,
                                                   **self.kw)
        loss = self.loss_fn(rgb, disp, acc, depth, extras, self.target, self.scale)
        loss.backward()                 # GradSync hooks (if any) start each network's allreduce as its gradients complete
        for sync in (self.sync, self.pose_sync):       # the networks' bucket, then the pose table's
            if sync is not None:
                sync.finish()
        return loss.detach()

    def _allreduce_eager(self):
        mdist.allreduce_grads(self.groups + ([self.pose_params] if self.pose_params else []))

    def _update(self):
        for opt in self.opts:
            opt.step_captured()
        for net in self.nets:                 # refresh the bf16 operand blobs the next forward reads
            net.repack()

    def _mark_packed_fresh(self):
        for net in self.nets:
            net._packed_key = net._pack_key(net._ordered_params())

    def capture(self):
        """Warm-up on a side stream (allocator pools, lazy module loads, smem opt-ins), then capture both graphs.  Parameters,
        Adam moments and the step count are snapshotted before and restored after the warm-up, so capturing trains nothing."""
        for opt in self.opts:
            opt.graph_begin(self.dev)
            opt.graph_set_lr()
        for net in run._net_params(self.kw):
            net[0].packed()
        params = [p for ps in self.groups for p in ps] + self.pose_params
        owner = [opt for opt in self.opts for g in opt.param_groups for _ in g["params"]]
        owned = [p for opt in self.opts for g in opt.param_groups for p in g["params"]]
        opt_of = {id(p): o for p, o in zip(owned, owner)}
        snap = [(p.detach().clone(), opt_of[id(p)].state[p]["exp_avg"].clone(), opt_of[id(p)].state[p]["exp_avg_sq"].clone())
                for p in params]
        step0 = [opt._g_step.clone() for opt in self.opts]
        s = torch.cuda.Stream(device=self.dev)
        s.wait_stream(torch.cuda.current_stream(self.dev))
        with torch.cuda.stream(s):
            for _ in range(self.warmup):
                self._forward_backward()
                if self.sync is None and self.pose_sync is None:
                    self._allreduce_eager()
                self._update()
                self._mark_packed_fresh()
        torch.cuda.current_stream(self.dev).wait_stream(s)
        torch.cuda.synchronize(self.dev)
        self.graph_a = torch.cuda.CUDAGraph()
        if self.one_graph:
            # NCCL's watchdog thread polls CUDA events while we capture: keep the capture thread-local
            mode = {"capture_error_mode": "thread_local"} if mdist.world() > 1 else {}
            with torch.cuda.graph(self.graph_a, **mode):
                self.loss = self._forward_backward()
                self._update()
        else:
            with torch.cuda.graph(self.graph_a):
                self.loss = self._forward_backward()
            self.graph_b = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph_b, pool=self.graph_a.pool()):
                self._update()
        with torch.no_grad():       # capture executes nothing; undo the warm-up steps
            for p, (w, m, v) in zip(params, snap):
                p.copy_(w)
                opt_of[id(p)].state[p]["exp_avg"].copy_(m)
                opt_of[id(p)].state[p]["exp_avg_sq"].copy_(v)
            for opt, st in zip(self.opts, step0):
                opt._g_step.copy_(st)
            for net in self.nets:
                net.repack()
        self._mark_packed_fresh()
        self._params = params
        self._static_grads = [p.grad for p in params]      # the buffers graph A writes and graph B / the allreduce read
        return self

    def __call__(self, rays=None, target=None):
        """One optimisation step; rays [2,N,3] (with `poses`: pixels [N,3] = (view, row, col), int32-representable) / target may
        be host (pinned) or device tensors, or None to reuse the buffers.
        Returns the loss of this step as a 0-dim device tensor (valid until the next call)."""
        if rays is not None:
            (self.rays if self.poses is None else self.pixels).copy_(rays, non_blocking=True)
        if target is not None:
            self.target.copy_(target, non_blocking=True)
        if self.graph_a is None:
            self.capture()
        for p, g in zip(self._params, self._static_grads):   # an eager backward in between may have re-pointed .grad
            if p.grad is not g:
                p.grad = g
        for opt in self.opts:
            opt.graph_set_lr()
        self.graph_a.replay()
        if self.graph_b is not None:
            self._allreduce_eager()
            self.graph_b.replay()
        for opt in self.opts:
            opt._g_dirty = True         # python-side step counts are refreshed lazily (FusedAdam.sync_graph_steps)
        return self.loss
