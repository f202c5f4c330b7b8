#!/usr/bin/env python
"""bench.py — headline measurement of the NeRF volume-rendering hot path on B200.

    python bench.py --gpus N --steps K --warmup W            # our arm (N>1: launched under torchrun)
    python bench.py --impl reference --gpus N --steps K --warmup W

metric  : rays/s of one training step (BASELINE.json cfg 2): N_rand = 4096 rays per GPU, 64 coarse +
          (64+64) fine samples, coarse+fine 8x256 MLP fwd+bwd, sample_pdf + raw2outputs, MSE loss on
          rgb and rgb0, gradient allreduce (N>1), Adam step.  Weak scaling: 4096 rays per GPU.
value   : whole-job rays/s with the ray batch already resident in HBM.
e2e     : the same step through the public API (mvip_nerf_b200.run.render) with HOST buffers: rays + targets
          copied from pinned memory every step, loss read back every step.
render  : secondary number — rendered rays/s of BASELINE.json cfg 3 (1008x756 image, render kwargs),
          rays sharded over the GPUs with one final gather.
roofline: the kernel with the largest share of the step, timed with CUDA events inside the timed region.
One JSON line on stdout (rank 0).

--dump-outputs DIR: after the timed steps, rank 0 writes what the last timed training step left its caller, as float32
DIR/<name>.npy: `loss` (the value the step returns), and for both networks `param.<net>.<tensor>` (the weights after that step's Adam update) and
`grad.<net>.<tensor>` (the gradients it applied), about 10 MB in all.  Rays, targets, initial weights and random draws are
seeded, so two builds run with the same arguments can be compared array for array.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

H, W, FOCAL, NEAR, FAR = 756, 1008, 767.2935, 1.2, 7.7369
N_RAND = 4096
METRIC = "rays/sec (train fwd+bwd, 64+64 samples)"
FLOP_FWD, FLOP_DGRAD, FLOP_WGRAD = 1186816, 1114112, 1185536       # per point, DESIGN.md §kernels
# HBM bytes per point: stash 40 chunk images x 128 B + 288 B masks; dZ stash 38 x 128 B (+ masks read, + 16 B d_raw);
# wgrad reads both sets of images; head grads read hidden (2) + h8 (4) images + d_raw
HBM_FWD_TRAIN, HBM_DGRAD, HBM_WGRAD, HBM_HEADS = 40 * 128 + 288 + 16, 38 * 128 + 288 + 16, 78 * 128, 6 * 128 + 16


def ncu_traffic(kernel, n_rand):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel`, from the committed `ncu --set full` capture of one
    cfg-2 step (profiles/ncu_traffic.json: written by scripts/summarize_profiles.py from the .ncu-rep; mean of the coarse
    and the fine launch), scaled to this run's rays per GPU.  None when the capture has no such kernel."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
        e = t["kernels"][kernel]
        return e["dram_bytes_per_launch"] * n_rand / t["rays_per_gpu"], t["source"]
    except Exception:
        return None, None


def workload_config(n_rand, world):
    """The `config` object: identical for the product arm and the reference arm (the driver compares them)."""
    return {"workload": ("cfg4" if n_rand * world == 65536 else "cfg2") +
            ": one training step, N_rand=%d rays per GPU, N_samples=64, N_importance=64, coarse+fine 8x256 NeRF (random init), "
            "lindisp, white_bkgd, perturb=1, raw_noise_std=1, loss=mse(rgb)+mse(rgb0), Adam" % n_rand,
            "rays_per_gpu": n_rand, "n_gpus": world, "parallelism": "rays sharded, dp%d, grad allreduce" % world,
            "l2": "no explicit flush between steps: every step streams ~8 GB of activation stash per GPU (>> 126 MB of L2)"}


def peaks():
    fallback = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "_source": "fallback"}
    try:
        d = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        d["_source"] = "measured"
        return d
    except Exception:
        return fallback


def nerf_args(basedir):
    return argparse.Namespace(
        multires=10, multires_views=4, i_embed=0, use_viewdirs=True, N_importance=64, N_samples=64, netdepth=8,
        netwidth=256, netdepth_fine=8, netwidth_fine=256, netchunk=65536, alpha_model_path=None, no_coarse=False,
        lrate=5e-4, basedir=basedir, expname="bench", ft_path=None, no_reload=True, perturb=1.0, white_bkgd=True,
        raw_noise_std=1.0, dataset_type="llff", no_ndc=True, lindisp=True, sigma_loss=False)


def synth_rays_np(n, seed):
    """cfg-2 rays: seeded random pixels of the 1008x756 pinhole grid, identity pose (SURVEY.md §8d)."""
    rng = np.random.RandomState(seed)
    idx = rng.randint(0, H * W, size=n)
    i = (idx % W).astype(np.float32)
    j = (idx // W).astype(np.float32)
    d = np.stack([(i - W * .5) / FOCAL, -(j - H * .5) / FOCAL, -np.ones_like(i)], -1).astype(np.float32)
    o = np.zeros_like(d)
    target = rng.rand(n, 3).astype(np.float32)
    return o, d, target


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def mark(self):
        """start of the timed region: samples before this instant are ignored"""
        self.t0 = time.time()

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        t_end = time.time()
        t0 = getattr(self, "t0", 0.0)
        for ts, ln in self.lines:
            if ts < t0 or ts > t_end:
                continue
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# =====================================================================================================
# reference arm: the UNMODIFIED reference (oracle/_ref or /root/reference) on the host cores; the CPU port only if the
# reference tree is not present
# =====================================================================================================
def host_threads():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def cpu_train_rays_per_s(n_rays, steps, warmup):
    """-> (rays/s, s/step, kind, threads): `steps` timed training steps of n_rays rays each, fp32, all host threads."""
    threads = host_threads()
    torch.set_num_threads(threads)          # torchrun exports OMP_NUM_THREADS=1: the CPU arm uses every core it may
    from oracle import ref_import
    o, d, target = synth_rays_np(n_rays, 1)
    if ref_import.available():
        run, helpers = ref_import.load()    # stock create_nerf + render + backward + torch.optim.Adam (run.py:914-1029)
        with tempfile.TemporaryDirectory() as td:
            os.makedirs(os.path.join(td, "bench"))
            torch.manual_seed(0)
            kw_train, _, _, _, opt = run.create_nerf(nerf_args(td))
        rays = torch.from_numpy(np.stack([o, d], 0))
        tgt = torch.from_numpy(target)

        def step():
            rgb, _, _, _, extras = run.render(H, W, FOCAL, chunk=32768, rays=rays, near=NEAR, far=FAR, **kw_train)
            opt.zero_grad()
            loss = helpers.img2mse(rgb, tgt) + helpers.img2mse(extras["rgb0"], tgt)
            loss.backward()
            opt.step()
        kind = "reference"
    else:
        from oracle import nerf_oracle as orc
        from oracle import torch_cpu_port as port
        pc = port.params_from_numpy(orc.init_params(1), True)
        pf = port.params_from_numpy(orc.init_params(2), True)
        rays = torch.from_numpy(orc.make_ray_batch(o, d, NEAR, FAR))
        tv = torch.linspace(0., 1., 64)
        g = torch.Generator().manual_seed(0)
        args = (torch.rand(n_rays, 64, generator=g), torch.rand(n_rays, 64, generator=g),
                torch.randn(n_rays, 64, generator=g), torch.randn(n_rays, 128, generator=g), torch.from_numpy(target))
        opt = torch.optim.Adam(list(pc.values()) + list(pf.values()), lr=5e-4)

        def step():
            port.train_step(rays, pc, pf, tv, *args)
            opt.step()
        kind = "port"
    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = time.perf_counter() - t0
    return n_rays * steps / dt, dt / steps, kind, threads


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sample = int(a.sample)
    val, sec, kind, threads = cpu_train_rays_per_s(sample, a.steps, a.warmup)
    what = ("the unmodified reference (DS_NeRF/run.py create_nerf + render + backward + torch.optim.Adam)" if kind == "reference"
            else "PyTorch-CPU port of the reference path (oracle/torch_cpu_port.py)")
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "rays/s", "n_gpus": a.gpus, "steps": a.steps,
            "warmup": a.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "fp32", "data": "synthetic", "config": workload_config(int(a.rays_per_gpu), a.gpus),
            "cpu_baseline": {"value": val, "unit": "rays/s", "cores": threads, "kind": kind,
                             "sample": "%d of the %d rays per step x %d steps, %s, fp32, %d threads"
                                       % (sample, int(a.rays_per_gpu), a.steps, what, threads)},
            "e2e": {"value": val, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def cpu_baseline_subprocess(sample, steps, warmup):
    """The same CPU arm from inside the product run: a child process with the GPUs hidden (the reference picks
    `cuda` when it sees one, run.py:46)."""
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "OMP_NUM_THREADS"):
        env.pop(k, None)
    p = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", str(steps), "--warmup", str(warmup),
                        "--sample", str(sample)], capture_output=True, text=True, timeout=900, env=env)
    for ln in p.stdout.splitlines():
        if ln.startswith("{"):
            return json.loads(ln)["cpu_baseline"]
    return {"value": None, "unit": "rays/s", "cores": 0, "kind": "unavailable", "sample": (p.stderr or "")[-200:]}


def hbm_stage_times(ops, dev, hbm_peak):
    """Sampling / compositing / ray / normal-map kernels on a 262,144-ray batch (a third of a cfg-3 image): achieved GB/s =
    ALGORITHMIC bytes per launch (SURVEY.md §8d, DESIGN.md §4.2) / CUDA-event time of the launch, best and median of 10."""
    N = 262144
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    g = torch.Generator(device=dev).manual_seed(0)
    rnd = lambda *sh: torch.rand(*sh, device=dev, generator=g)  # noqa: E731

    def timeit(fn):
        for _ in range(3):
            fn()
        ts = []
        for _ in range(10):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); fn(); b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        return float(np.median(ts)), float(np.min(ts))
    out = {}

    def add(name, nbytes, fn):
        med, best = timeit(fn)
        out[name] = {"bytes_per_launch": nbytes, "ms_median": med, "ms_best": best, "gbs": nbytes / med / 1e6,
                     "frac_of_hbm_peak": nbytes / med / 1e6 / hbm_peak}
    for S in (64, 128):
        raw = rnd(N, S, 4) * 2 - 1
        z = torch.sort(rnd(N, S) * 6 + 1.2, -1)[0]
        rd = rnd(N, 3) - .5
        add("composite_fwd_S%d" % S, N * (S * 20 + 12 + S * 4 + 24), lambda: ops.composite_forward(raw, z, rd, None, True))
        gs = [rnd(N, 3), rnd(N), rnd(N), rnd(N)]
        add("composite_bwd_S%d" % S, N * (S * 20 + 12 + 24 + S * 16), lambda: ops.composite_backward(raw, z, rd, None, True, False, *gs))
    z = torch.sort(rnd(N, 64) * 6 + 1.2, -1)[0]
    w = rnd(N, 64) ** 4
    u = rnd(N, 64)
    add("sample_fine_rand_u", N * (512 + 256 + 512 + 4), lambda: ops.sample_fine(z, w, u, want_samples=False))
    rays = rnd(N, 11) + 1
    tv = torch.linspace(0, 1, 64, device=dev)
    tr = rnd(N, 64)
    add("sample_coarse_perturb", N * (8 + 256 + 256), lambda: ops.sample_coarse(rays, tv, tr, True))
    c2w = torch.eye(4, device=dev)[:3, :4].contiguous()
    add("rays_from_pose_1008x756", H * W * 44, lambda: ops.rays_from_pose(H, W, FOCAL, c2w, NEAR, FAR))
    d = rnd(512, 512) + 3
    add("normal_fwd_512x512_k31", 512 * 512 * 24, lambda: ops.normal_forward(d, 500., 500., 256., 256., 31))
    return out


# =====================================================================================================
# our arm
# =====================================================================================================
# kernel label (ops.kernel_timer) -> (FLOP per point, algorithmic HBM bytes per point, direction)
def kernel_table():
    return {"mvip_mlp_forward": (FLOP_FWD, HBM_FWD_TRAIN, "write"),
            # fused backward (dgrad chain + all weight gradients): dZ is written once (and re-read out of L2 by the wgrad role),
            # the forward stash is read once
            "backward_fused_kernel": (FLOP_DGRAD + FLOP_WGRAD, HBM_DGRAD + 40 * 128, "read+write"),
            "head_grads_kernel": (0, HBM_HEADS, "read")}


def dump_outputs(out_dir, loss, nets):
    """--dump-outputs: the loss of the last step and, per network, its updated parameters and the gradients it applied."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"loss": loss}
    for net_name, net in nets.items():
        for name, p in net.named_parameters():
            name = net_name + "." + name.replace("module.", "")
            arrays["param." + name] = p
            arrays["grad." + name] = p.grad
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().float().cpu().numpy())


def run_ours(a):
    global N_RAND
    N_RAND = int(a.rays_per_gpu)
    from mvip_nerf_b200 import dist as md
    from mvip_nerf_b200 import ops, run
    from mvip_nerf_b200.run_nerf_helpers import img2mse
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the product path has no CPU fallback (use --impl reference for the CPU arm)")
    rank, world, local = md.init_from_env()
    dev = torch.device("cuda", local)
    pk = peaks()

    with tempfile.TemporaryDirectory() as td:
        os.makedirs(os.path.join(td, "bench"))
        torch.manual_seed(0)
        kw_train, kw_test, _, grad_vars, optimizer = run.create_nerf(nerf_args(td))   # optimizer: FusedAdam (one launch)
    coarse, fine = kw_train["network_fn"], kw_train["network_fine"]
    groups = [list(fine.parameters()), list(coarse.parameters())]
    inv_world = 1.0 / world
    sync = md.GradSync(groups, overlap=a.overlap_allreduce)

    def step(rays, tgt):
        optimizer.zero_grad(set_to_none=True)
        rgb, disp, acc, depth, extras = run.render(H, W, FOCAL, chunk=32768, rays=rays, near=NEAR, far=FAR, **kw_train)
        loss = (img2mse(rgb, tgt) + img2mse(extras["rgb0"], tgt)) * inv_world     # mean over the GLOBAL batch
        loss.backward()
        sync.finish()
        optimizer.step()
        return loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    def make_batch(n_rand):
        o, d, target = synth_rays_np(n_rand, 100 + rank)
        pin = lambda x: torch.from_numpy(x).pin_memory()  # noqa: E731
        h_rays, h_t = pin(np.stack([o, d], 0)), pin(target)
        return h_rays, h_t, h_rays.to(dev), h_t.to(dev)

    def make_graphed(n_rand, d_rays, d_target):
        """the step as the product runs it (graph.GraphedTrainStep): ONE CUDA graph incl. the NCCL buckets; if NCCL refuses to be
        captured: two graphs with the eager allreduce between them; eager launches if capture fails altogether"""
        if a.no_graph:
            return None, "eager launches"
        from mvip_nerf_b200.graph import GraphedTrainStep
        for in_graph, note in ((True, "one CUDA graph per step: render + loss + backward + ONE NCCL allreduce of both networks' gradients + Adam + bf16 re-pack"),
                               (False, "two CUDA graphs per step: (render + loss + backward) | eager NCCL allreduce | (Adam + bf16 re-pack)")):
            if not in_graph and world == 1:
                break
            try:
                g = GraphedTrainStep(kw_train, optimizer, H, W, FOCAL, n_rand, NEAR, FAR, nccl_in_graph=in_graph, overlap_allreduce=a.overlap_allreduce)
                g.rays.copy_(d_rays)
                g.target.copy_(d_target)
                g.capture()
                return g, note
            except Exception as e:      # noqa: BLE001
                err = str(e)[:160]
                torch.cuda.synchronize()
        return None, "eager launches (graph capture failed: %s)" % err

    h_rays, h_t, d_rays, d_target = make_batch(N_RAND)
    sync.remove()                       # GraphedTrainStep installs its own hooks; the eager region below re-installs these
    gstep, graph_note = make_graphed(N_RAND, d_rays, d_target)

    def resident_step():
        return gstep() if gstep is not None else step(d_rays, d_target)

    # ---- device-resident arm ---------------------------------------------------------------------
    if gstep is None:
        sync = md.GradSync(groups, overlap=a.overlap_allreduce)
    for _ in range(a.warmup):
        resident_step()
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    for _ in range(3):                         # nvidia-smi needs ~100 ms to start streaming: keep the GPUs busy meanwhile
        resident_step()                        # (all ranks: the step contains a collective)
    torch.cuda.synchronize()
    clocks.mark()
    last = {}

    def timed_step():
        last["loss"] = resident_step()
    ms_total = timed(timed_step, a.steps)
    clk = clocks.stop() if rank == 0 else None
    if a.dump_outputs and rank == 0:       # before the sections below train the networks further
        dump_outputs(a.dump_outputs, last["loss"], {"coarse": coarse, "fine": fine})
    ms_step = ms_total / a.steps
    value = world * N_RAND / (ms_step * 1e-3)

    # ---- end-to-end arm: host buffers, H2D every step, loss read back every step -----------------------
    def e2e_step():
        if gstep is not None:
            return float(gstep(h_rays, h_t).item())
        return float(step(h_rays.to(dev, non_blocking=True), h_t.to(dev, non_blocking=True)).item())
    for _ in range(max(1, a.warmup // 2)):
        e2e_step()
    ms_e2e = timed(e2e_step, a.steps) / a.steps
    e2e_value = world * N_RAND / (ms_e2e * 1e-3)

    # ---- secondary (8 GPUs): BASELINE cfg 4, N_rand = 65,536 rays per step = 8,192 per GPU ------------------------
    cfg4 = None
    if world == 8 and N_RAND != 8192:
        if gstep is not None and gstep.sync is not None:
            gstep.sync.remove()
        b4 = make_batch(8192)
        g4, _ = make_graphed(8192, b4[2], b4[3])
        if g4 is not None:
            for _ in range(3):
                g4()
            ms4 = timed(g4, a.steps) / a.steps
            cfg4 = {"rays_s": world * 8192 / (ms4 * 1e-3), "ms_per_step": ms4, "global_rays": 65536}
            if g4.sync is not None:
                g4.sync.remove()
            del g4
    elif gstep is not None and gstep.sync is not None:
        gstep.sync.remove()

    # ---- the same K steps launched eagerly with a CUDA-event bracket around every library call: per-kernel times --------
    sync = md.GradSync(groups, overlap=a.overlap_allreduce)
    for _ in range(3):
        step(d_rays, d_target)
    ops.kernel_timer.enable(True)
    l0 = ops.launch_count
    ms_eager = timed(lambda: step(d_rays, d_target), a.steps) / a.steps
    launches = ops.launch_count - l0
    ktimes = ops.kernel_timer.collect()
    ops.kernel_timer.enable(False)
    sync.remove()

    # ---- secondary: full-image render (cfg 3), rays sharded, one gather ------------------------------
    n_img = H * W
    c2w = torch.eye(4, device=dev)[:3, :4]
    rays_flat = ops.rays_from_pose(H, W, FOCAL, c2w, NEAR, FAR, use_viewdirs=True, ndc=False)
    kw_r = {k: v for k, v in kw_test.items() if k not in ("ndc", "use_viewdirs")}

    def render_image():
        with torch.no_grad():
            return md.render_sharded(lambda rows: run.batchify_rays(rows, 1 << 17, **kw_r), rays_flat)
    render_image()
    r_steps = 3
    ms_render = timed(render_image, r_steps) / r_steps
    render_value = n_img / (ms_render * 1e-3)

    # ---- secondary: guidance batch (cfg 5): 4 views x 512 x 512, rgb + disp + acc + depth, normal maps on rank 0 --------
    GV, GH, GW = 4, 512, 512
    gfocal = FOCAL * GW / W
    gposes = []
    for v in range(GV):
        pz = torch.eye(4, device=dev)[:3, :4].clone()
        pz[0, 3] = 0.1 * v
        gposes.append(pz)

    def render_nograd(*args, **kw):
        with torch.no_grad():
            return run.render(*args, chunk=1 << 17, **kw)

    def guidance():
        return md.render_views_sharded(render_nograd, gposes, GH, GW, gfocal, NEAR, FAR, **kw_test)
    guidance()
    g_steps = 2
    ms_guid = timed(guidance, g_steps) / g_steps
    guid_value = GV * GH * GW / (ms_guid * 1e-3)

    # ---- secondary: one guidance view WITH gradients at full resolution (deferred back-propagation, SURVEY §8 f2) --------
    # every rank renders its own 512 x 512 view (render kwargs), image loss on rgb + depth, backward through render_deferred
    def guidance_train():
        optimizer.zero_grad(set_to_none=True)
        rgb, disp, acc, depth, _ = run.render_deferred(GH, GW, gfocal, chunk=8192, c2w=gposes[rank % GV], near=NEAR, far=FAR, **kw_test)
        loss = ((rgb - 0.5) ** 2).mean() + 0.1 * depth.mean()
        loss.backward()
    guidance_train()
    ms_gtrain = timed(guidance_train, 1)
    gtrain_value = world * GH * GW / (ms_gtrain * 1e-3)

    if rank != 0:
        finish_process(world)
        return

    # ---- HBM-bound stages at image-sized batches (rank 0, CUDA events per launch, L2 flushed between launches) ---------
    # These kernels are timed ALONE against the burst copy peak: let the board leave the power-capped state the render /
    # guidance sections above put it in (measured: the same kernels reach 0.87 of the peak on an idle GPU, 0.70 right after them).
    torch.cuda.synchronize()
    time.sleep(2.0)
    hbm_stages = hbm_stage_times(ops, dev, pk["hbm_gbs"])

    # ---- per-kernel rooflines (CUDA events around each launch of the eager region) -----------------------------------------
    # Tensor denominators: the cuBLAS bf16 burst peak for a timed region under 1 s (the clocks have not settled under the
    # power cap: this is the honest roof for a 20-step run), the sustained peak for a longer one; both fractions are printed.
    npts = N_RAND * 192
    tf_burst, tf_sust = pk["bf16_tflops"], pk.get("bf16_tflops_sustained", pk["bf16_tflops"])
    short = ms_total < 1000.0
    peak_tf = tf_burst if short else tf_sust
    table = kernel_table()
    per_kernel = {}
    for name, vals in ktimes.items():
        ms_k = sum(vals) / a.steps
        e = {"launches_per_step": len(vals) / a.steps, "ms_per_step": ms_k, "share_of_step": ms_k / ms_eager}
        if name in table:
            fl, by, kind = table[name]
            if fl:
                e["tflops"] = fl * npts / (ms_k * 1e-3) / 1e12
                e["frac_of_tensor_burst"], e["frac_of_tensor_sustained"] = e["tflops"] / tf_burst, e["tflops"] / tf_sust
            e["hbm_gbs"] = by * npts / (ms_k * 1e-3) / 1e9
            e["frac_of_hbm_peak"] = e["hbm_gbs"] / pk["hbm_gbs"]
            e["hbm_direction"] = kind
        per_kernel[name] = e
    mlp_kernels = [k for k in per_kernel if k in table and table[k][0]]
    top = max(mlp_kernels, key=lambda k: per_kernel[k]["ms_per_step"]) if mlp_kernels else None
    roofline = None
    if top:
        e = per_kernel[top]
        traffic, traffic_src = ncu_traffic(top, N_RAND)
        roofline = {"kernel": top, "bound": "tensor", "achieved": e["tflops"], "peak": peak_tf, "unit": "TFLOP/s",
                    "frac": e["tflops"] / peak_tf, "frac_burst": e["frac_of_tensor_burst"], "frac_sustained": e["frac_of_tensor_sustained"],
                    "peak_source": "%s cuBLAS bf16 %s peak (timed region %.0f ms)" % (pk["_source"], "burst" if short else "sustained", ms_total),
                    "traffic": traffic, "traffic_source": traffic_src,
                    "share_of_step": e["share_of_step"],
                    "hbm": {"achieved": e["hbm_gbs"], "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": e["frac_of_hbm_peak"],
                            "direction": e["hbm_direction"], "algorithmic_bytes_per_launch": table[top][1] * npts / 2,
                            "note": "the design moves the activation / dZ stash through HBM (DESIGN.md §3); §8(d)'s algorithmic "
                                    "work of the MLP is FLOPs, hence bound=tensor and this figure beside it"}}
    train_tf = world * N_RAND * 192 * (FLOP_FWD + FLOP_DGRAD + FLOP_WGRAD) / (ms_step * 1e-3) / 1e12
    render_tf = n_img * 192 * FLOP_FWD / (ms_render * 1e-3) / 1e12
    if roofline is not None:     # compact secondaries: the driver keeps `roofline` / `e2e` / `config` of the line, not extra keys
        roofline["step"] = {"train_tflops": train_tf, "frac_burst": train_tf / (tf_burst * world), "frac_sustained": train_tf / (tf_sust * world)}
        roofline["secondary"] = {
            "render_cfg3_rays_s": render_value, "render_tflops": render_tf, "render_frac_burst": render_tf / (tf_burst * world),
            "render_frac_sustained": render_tf / (tf_sust * world), "guidance_cfg5_rays_s": guid_value,
            "guidance_train_rays_s": gtrain_value, "train_cfg4_rays_s": cfg4["rays_s"] if cfg4 else None,
            "composite_fwd_S128_frac_hbm": hbm_stages["composite_fwd_S128"]["frac_of_hbm_peak"],
            "composite_bwd_S128_frac_hbm": hbm_stages["composite_bwd_S128"]["frac_of_hbm_peak"],
            "sample_fine_frac_hbm": hbm_stages["sample_fine_rand_u"]["frac_of_hbm_peak"],
            "sample_coarse_frac_hbm": hbm_stages["sample_coarse_perturb"]["frac_of_hbm_peak"]}

    # ---- CPU baseline on the host cores (bounded sample; child process with the GPUs hidden) ----------------------------
    cpu_base = None
    if world == 1 and not a.no_cpu_baseline:
        cpu_base = cpu_baseline_subprocess(1024, 8, 1)

    bytes_in = (h_rays.numel() + h_t.numel()) * 4
    line = {
        "metric": METRIC, "value": value, "unit": "rays/s", "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
        "data": "synthetic",
        "config": workload_config(N_RAND, world),
        "e2e": {"value": e2e_value, "unit": "rays/s", "h2d_bytes_per_step": bytes_in, "d2h_bytes_per_step": 4,
                "ms_per_step": ms_e2e},
        "gpu_launches": launches,
        "clocks": clk,
        "roofline": roofline,
        "notes": {"launch": graph_note,
                  "kernel_times": "CUDA events around every library call in a second timed region of the same %d steps launched "
                                  "eagerly (%.3f ms/step); gpu_launches counts that region" % (a.steps, ms_eager),
                  "l2": "no explicit flush: each step streams ~8 GB of activation stash per GPU (>> 126 MB L2)"},
        "kernels": per_kernel,
        "render": {"value": render_value, "unit": "rays/s", "ms_per_image": ms_render,
                   "workload": "cfg3: 1008x756 image (762,048 rays), render kwargs, rays sharded over %d GPU(s), one gather" % world,
                   "tflops": render_tf, "bound": "tensor"},
        "guidance": {"value": guid_value, "unit": "rays/s", "ms_per_batch": ms_guid,
                     "workload": "cfg5: %d views of %dx%d (rgb + disp + acc + depth), image rows sharded over %d GPU(s), one gather, "
                                 "normal maps (k=31) of all views on rank 0" % (GV, GH, GW, world)},
        "guidance_train": {"value": gtrain_value, "unit": "rays/s", "ms_per_view": ms_gtrain,
                           "workload": "one 512x512 view per GPU, forward + image loss + deferred back-propagation "
                                       "(re-render in 8192-ray chunks), parameter gradients of both networks"},
        "train_cfg4": cfg4,
        "hbm_stages": hbm_stages,
        "train_tflops": train_tf,
    }
    if cpu_base is not None:
        line["cpu_baseline"] = cpu_base
    print(json.dumps(line), flush=True)
    finish_process(world)


def finish_process(world):
    """End of a rank under torchrun.  destroy_process_group() can block for minutes while captured CUDA graphs still hold NCCL
    work (seen on 2 B200: the JSON line was out, the launcher only returned when its timeout fired); every result has been
    printed and flushed at this point, so the rank leaves without running NCCL's teardown."""
    if world > 1:
        torch.cuda.synchronize()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--rays-per-gpu", type=int, default=N_RAND,
                    help="N_rand per GPU: 4096 = BASELINE cfg 2 (default, the configuration `metric` is quoted on); 8192 with "
                         "--gpus 8 = cfg 4 (65,536 rays per step; also measured as a secondary entry of every 8-GPU run)")
    ap.add_argument("--sample", type=int, default=1024,
                    help="reference arm: rays per timed step (a bounded sample of the N_rand batch; 1024 = the reference's own N_rand)")
    ap.add_argument("--overlap-allreduce", action="store_true",
                    help="start each network's gradient allreduce from autograd hooks while the backward still runs (default: after it)")
    ap.add_argument("--no-graph", action="store_true", help="launch the step eagerly instead of replaying CUDA graphs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the loss, parameters and gradients of the last timed step to DIR/<name>.npy (product arm)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.impl == "reference":
        if a.dump_outputs:
            ap.error("--dump-outputs writes what the product arm computed; the reference arm has none")
        os.environ["CUDA_VISIBLE_DEVICES"] = ""      # the reference picks `cuda` when it sees one (run.py:46): this arm is its CPU path
        run_reference(a)
    else:
        a.warmup = max(a.warmup, 3)
        run_ours(a)


if __name__ == "__main__":
    main()
