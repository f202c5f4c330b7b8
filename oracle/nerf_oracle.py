"""CPU oracle for the MVIP-NeRF volume-rendering hot path — TEST INFRASTRUCTURE ONLY.

This file is a numpy restatement of the reference's algorithm (DS_NeRF/run.py,
DS_NeRF/run_nerf_helpers.py); it is the checker for the CUDA path, never the
product.  Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
--impl reference legs may import it.  mvip_nerf_b200/ never does.

Parity pinning: the reference ships no golden vectors for this path (SURVEY.md
§8c), so the oracle is pinned against the reference *executed* in the build
container: oracle/make_golden.py imports /root/reference (oracle/ref_import.py),
runs the reference functions on seeded inputs and commits inputs+outputs under
tests/golden/; tests/test_oracle_golden.py replays them through this file.
Bit-exact stages (coarse z, cdf, inds, samples, merged z) are compared with ==.

Every function cites the reference lines it follows (paths relative to
/root/reference/).  All arithmetic is float32 unless a comment says otherwise.
"""
import numpy as np

f32 = np.float32


# --------------------------------------------------------------------------------------
# small helpers that pin third-party (PyTorch CPU) rounding behaviour
# --------------------------------------------------------------------------------------
def linspace_f32(start, end, steps):
    """torch.linspace(start, end, steps) for float32 on CPU (ATen RangeFactories):
    step=(end-start)/(steps-1) in float32; the first half is fma(step, i, start), the
    second half fma(-step, steps-1-i, end) (the float64 product of two float32 values is
    exact, so the float64 expression below rounds once, like the fused op).  Verified ==
    torch.linspace for steps in {2..1000}.  Used for t_vals (run.py:1759) and the
    deterministic u (run_nerf_helpers.py:313)."""
    start = f32(start)
    end = f32(end)
    if steps == 1:
        return np.array([start], dtype=f32)
    step = f32((end - start) / f32(steps - 1))
    i = np.arange(steps)
    lo = (np.float64(start) + np.float64(step) * i).astype(f32)
    hi = (np.float64(end) - np.float64(step) * (steps - 1 - i)).astype(f32)
    return np.where(i < steps // 2, lo, hi).astype(f32)


def aten_sum_lastdim(x):
    """torch.sum(x, -1) for contiguous float32 rows on CPU, in ATen's exact order
    (SURVEY.md §8a): 8 SIMD lanes x 4 interleaved accumulators, leftover vectors into
    accumulator 0, accumulators combined 0+1+2+3, then the scalar tail summed
    sequentially starting from 0 and finally the 8 lanes added in lane order.
    Pins `torch.sum(weights, -1, keepdim=True)` of run_nerf_helpers.py:307."""
    x = np.ascontiguousarray(x, dtype=f32)
    K = x.shape[-1]
    if 5 <= K <= 7 or K > 512:
        raise ValueError("aten_sum_lastdim restatement verified only for K in [1,4] U [8,512] (got %d)" % K)
    lead = x.shape[:-1]
    x2 = x.reshape(-1, K)
    nv = K // 8
    nfull = 4 * (nv // 4)
    ps = [np.zeros((x2.shape[0], 8), dtype=f32) for _ in range(4)]
    started = [False] * 4
    for v in range(nfull):
        blk = x2[:, 8 * v:8 * v + 8]
        u = v % 4
        ps[u] = blk.copy() if not started[u] else (ps[u] + blk).astype(f32)
        started[u] = True
    for v in range(nfull, nv):
        blk = x2[:, 8 * v:8 * v + 8]
        ps[0] = blk.copy() if not started[0] else (ps[0] + blk).astype(f32)
        started[0] = True
    if nfull > 0:
        t = (ps[0] + ps[1]).astype(f32)
        t = (t + ps[2]).astype(f32)
        t = (t + ps[3]).astype(f32)
    else:
        t = ps[0]
    acc = np.zeros(x2.shape[0], dtype=f32)
    for k in range(8 * nv, K):
        acc = (acc + x2[:, k]).astype(f32)
    if nv > 0:
        for lane in range(8):
            acc = (acc + t[:, lane]).astype(f32)
    return acc.reshape(lead)


def cumsum_f64_round_f32(x):
    """torch.cumsum(x, -1) for float32 on CPU: sequential accumulation in float64,
    rounded to float32 at every output (SURVEY.md §8a; run_nerf_helpers.py:308)."""
    return np.cumsum(x.astype(np.float64), axis=-1).astype(f32)


def cumprod_f64_round_f32(x):
    """torch.cumprod(x, -1) for float32 on CPU: float64 accumulation, float32 outputs
    (run_nerf_helpers.py:385)."""
    return np.cumprod(x.astype(np.float64), axis=-1).astype(f32)


# --------------------------------------------------------------------------------------
# a3: stratified sampling   (run.py:1750-1784)
# --------------------------------------------------------------------------------------
def sample_coarse(rays, t_vals, t_rand=None, lindisp=False):
    """rays [N,>=8] (o,d,near,far,...), t_vals [S] table (torch.linspace on the host),
    t_rand [N,S] or None (perturb==0).  Returns z_vals [N,S].  Every op rounds to
    float32, no FMA contraction (numpy never fuses)."""
    rays = np.asarray(rays, dtype=f32)
    near = rays[:, 6:7]
    far = rays[:, 7:8]
    t = np.asarray(t_vals, dtype=f32)[None, :]
    one = f32(1.0)
    if not lindisp:
        z = (near * (one - t)).astype(f32) + (far * t).astype(f32)          # run.py:1761
    else:
        a = (one / near).astype(f32)
        b = (one / far).astype(f32)
        den = ((a * (one - t)).astype(f32) + (b * t).astype(f32)).astype(f32)
        z = (one / den).astype(f32)                                          # run.py:1763
    z = np.broadcast_to(z.astype(f32), (rays.shape[0], t.shape[1])).copy()
    if t_rand is not None:
        mids = (f32(0.5) * (z[:, 1:] + z[:, :-1]).astype(f32)).astype(f32)   # run.py:1769
        upper = np.concatenate([mids, z[:, -1:]], -1)
        lower = np.concatenate([z[:, :1], mids], -1)
        z = (lower + ((upper - lower).astype(f32) * np.asarray(t_rand, dtype=f32)).astype(f32)).astype(f32)  # :1781
    return z


def points(rays, z):
    """pts = o + d*z (run.py:1783), separate multiply and add."""
    o = rays[:, None, 0:3].astype(f32)
    d = rays[:, None, 3:6].astype(f32)
    return (o + (d * z[:, :, None]).astype(f32)).astype(f32)


# --------------------------------------------------------------------------------------
# a8: sample_pdf   (run_nerf_helpers.py:304-347)
# --------------------------------------------------------------------------------------
def sample_pdf(bins, weights, u):
    """bins [N,B], weights [N,B-1], u [N,M] (host-provided: torch.linspace row for det,
    uniform randoms otherwise).  Returns dict(cdf [N,B], inds [N,M] int64, samples [N,M])."""
    bins = np.asarray(bins, dtype=f32)
    w = (np.asarray(weights, dtype=f32) + f32(1e-5)).astype(f32)              # :306
    s = aten_sum_lastdim(w)[:, None]
    pdf = (w / s).astype(f32)                                                 # :307
    cdf = cumsum_f64_round_f32(pdf)                                           # :308
    cdf = np.concatenate([np.zeros_like(cdf[:, :1]), cdf], -1)                # :309
    u = np.ascontiguousarray(np.broadcast_to(np.asarray(u, dtype=f32), (bins.shape[0], np.shape(u)[-1])))
    N, M = u.shape
    B = cdf.shape[-1]
    inds = np.empty((N, M), dtype=np.int64)
    for r in range(N):                                                        # :331 searchsorted(right=True)
        inds[r] = np.searchsorted(cdf[r], u[r], side="right")
    below = np.maximum(0, inds - 1)                                           # :332
    above = np.minimum(B - 1, inds)                                           # :333
    cdf_b = np.take_along_axis(cdf, below, 1)
    cdf_a = np.take_along_axis(cdf, above, 1)
    bins_b = np.take_along_axis(bins, below, 1)
    bins_a = np.take_along_axis(bins, above, 1)
    denom = (cdf_a - cdf_b).astype(f32)                                       # :342
    denom = np.where(denom < f32(1e-5), f32(1.0), denom).astype(f32)          # :343
    t = ((u - cdf_b).astype(f32) / denom).astype(f32)                         # :344
    samples = (bins_b + (t * (bins_a - bins_b).astype(f32)).astype(f32)).astype(f32)  # :345
    return {"cdf": cdf, "inds": inds, "below": below, "above": above, "samples": samples}


def fine_samples(z_vals, weights, u):
    """run.py:1809-1816: z_mid, sample_pdf on weights[...,1:-1], sort(cat).  Returns
    dict(z_samples, inds, z_merged, z_std)."""
    z_vals = np.asarray(z_vals, dtype=f32)
    z_mid = (f32(0.5) * (z_vals[:, 1:] + z_vals[:, :-1]).astype(f32)).astype(f32)   # :1809
    sp = sample_pdf(z_mid, np.asarray(weights, dtype=f32)[:, 1:-1], u)              # :1810
    z_samples = sp["samples"]
    z_merged = np.sort(np.concatenate([z_vals, z_samples], -1), -1)                 # :1814
    # torch.std(unbiased=False) (run.py:1836): float32 two-pass; compared with tolerance
    z_std = np.std(z_samples.astype(np.float64), axis=-1).astype(f32)
    return {"z_samples": z_samples, "inds": sp["inds"], "cdf": sp["cdf"],
            "z_merged": z_merged, "z_std": z_std}


# --------------------------------------------------------------------------------------
# a5: positional encoding   (run_nerf_helpers.py:22-70)
# --------------------------------------------------------------------------------------
def embed(x, num_freqs):
    """[x, sin(x*1), cos(x*1), sin(x*2), cos(x*2), ...] with freq = 2**k exact powers of
    two (log_sampling, :39); output dim 3 + 6*num_freqs."""
    x = np.asarray(x, dtype=f32)
    outs = [x]
    for k in range(num_freqs):
        xf = (x * f32(2.0 ** k)).astype(f32)
        outs.append(np.sin(xf).astype(f32))
        outs.append(np.cos(xf).astype(f32))
    return np.concatenate(outs, -1)


# --------------------------------------------------------------------------------------
# a6: NeRF MLP   (run_nerf_helpers.py:74-127), use_viewdirs=True, skips=[4]
# --------------------------------------------------------------------------------------
PARAM_NAMES = (["pts_linears.%d" % i for i in range(8)] +
               ["views_linears.0", "feature_linear", "alpha_linear", "rgb_linear"])


def init_params(seed, D=8, W=256, input_ch=63, input_ch_views=27, skips=(4,), dtype=f32):
    """nn.Linear-style uniform(-1/sqrt(fan_in), 1/sqrt(fan_in)) init from numpy's frozen
    legacy MT19937 stream (RandomState), so fixtures need not store the 2.4 MB of weights:
    make_golden.py loads exactly these values into the reference's NeRF modules."""
    rng = np.random.RandomState(seed)
    shapes = {}
    shapes["pts_linears.0"] = (W, input_ch)
    for i in range(1, D):
        shapes["pts_linears.%d" % i] = (W, W + input_ch) if (i - 1) in skips else (W, W)
    shapes["views_linears.0"] = (W // 2, input_ch_views + W)
    shapes["feature_linear"] = (W, W)
    shapes["alpha_linear"] = (1, W)
    shapes["rgb_linear"] = (3, W // 2)
    p = {}
    for name, (o, i) in shapes.items():
        bound = 1.0 / np.sqrt(i)
        p[name + ".weight"] = rng.uniform(-bound, bound, size=(o, i)).astype(dtype)
        p[name + ".bias"] = rng.uniform(-bound, bound, size=(o,)).astype(dtype)
    return p


def nerf_forward(p, x, D=8, skips=(4,), input_ch=63, keep=False, dtype=f32):
    """NeRF.forward (run_nerf_helpers.py:104-127) on x [P, 63+27] -> [P,4] = (rgb, alpha).
    With keep=True also returns the layer inputs/outputs needed by nerf_backward."""
    x = np.asarray(x, dtype=dtype)
    pts, views = x[:, :input_ch], x[:, input_ch:]
    h = pts
    saved = {"ins": [], "pre": []}
    for i in range(D):
        saved["ins"].append(h)
        pre = h @ p["pts_linears.%d.weight" % i].T.astype(dtype) + p["pts_linears.%d.bias" % i].astype(dtype)
        saved["pre"].append(pre)
        h = np.maximum(pre, 0)                                                # :108-109
        if i in skips:
            h = np.concatenate([pts, h], -1)                                  # :110-111
    alpha = h @ p["alpha_linear.weight"].T.astype(dtype) + p["alpha_linear.bias"].astype(dtype)      # :114
    feature = h @ p["feature_linear.weight"].T.astype(dtype) + p["feature_linear.bias"].astype(dtype)  # :115
    hv_in = np.concatenate([feature, views], -1)                              # :116
    pre_v = hv_in @ p["views_linears.0.weight"].T.astype(dtype) + p["views_linears.0.bias"].astype(dtype)
    hv = np.maximum(pre_v, 0)                                                 # :119-120
    rgb = hv @ p["rgb_linear.weight"].T.astype(dtype) + p["rgb_linear.bias"].astype(dtype)             # :122
    out = np.concatenate([rgb, alpha], -1).astype(dtype)                      # :123
    if keep:
        saved.update(h8=h, hv_in=hv_in, pre_v=pre_v, hv=hv)
        return out, saved
    return out


def nerf_backward(p, saved, d_out, D=8, skips=(4,), input_ch=63, dtype=f32):
    """Gradients of all parameters for upstream d_out [P,4] (what autograd computes for
    NeRF.forward).  No gradient flows to the inputs (pts/views are not leaves that
    require grad in the reference: z_samples is detached, run.py:1812)."""
    g = {}
    d_out = np.asarray(d_out, dtype=dtype)
    d_rgb, d_alpha = d_out[:, :3], d_out[:, 3:4]
    g["rgb_linear.weight"] = d_rgb.T @ saved["hv"]
    g["rgb_linear.bias"] = d_rgb.sum(0)
    d_hv = d_rgb @ p["rgb_linear.weight"].astype(dtype)
    d_pre_v = d_hv * (saved["pre_v"] > 0)
    g["views_linears.0.weight"] = d_pre_v.T @ saved["hv_in"]
    g["views_linears.0.bias"] = d_pre_v.sum(0)
    W = p["feature_linear.weight"].shape[0]
    d_feature = (d_pre_v @ p["views_linears.0.weight"].astype(dtype))[:, :W]
    g["feature_linear.weight"] = d_feature.T @ saved["h8"]
    g["feature_linear.bias"] = d_feature.sum(0)
    g["alpha_linear.weight"] = d_alpha.T @ saved["h8"]
    g["alpha_linear.bias"] = d_alpha.sum(0)
    d_h = d_feature @ p["feature_linear.weight"].astype(dtype) + d_alpha @ p["alpha_linear.weight"].astype(dtype)
    for i in reversed(range(D)):
        if i in skips:
            d_h = d_h[:, input_ch:]            # the cat([pts, h]) of :111 — drop the pts columns
        d_pre = d_h * (saved["pre"][i] > 0)
        g["pts_linears.%d.weight" % i] = d_pre.T @ saved["ins"][i]
        g["pts_linears.%d.bias" % i] = d_pre.sum(0)
        d_h = d_pre @ p["pts_linears.%d.weight" % i].astype(dtype)
    return {k: v.astype(dtype) for k, v in g.items()}


def run_network(p, pts, viewdirs, multires=10, multires_views=4, keep=False, dtype=f32):
    """run.py:1108-1124: flatten, embed pts and (expanded) viewdirs, cat, MLP, reshape."""
    N, S, _ = pts.shape
    flat = pts.reshape(-1, 3)
    e = embed(flat, multires)
    dirs = np.broadcast_to(viewdirs[:, None, :], pts.shape).reshape(-1, 3)
    ed = embed(dirs, multires_views)
    x = np.concatenate([e, ed], -1).astype(dtype)
    if keep:
        out, saved = nerf_forward(p, x, keep=True, dtype=dtype)
        return out.reshape(N, S, 4), saved
    return nerf_forward(p, x, dtype=dtype).reshape(N, S, 4)


# --------------------------------------------------------------------------------------
# a7: raw2outputs   (run_nerf_helpers.py:350-404) + hand-derived backward (SURVEY §8a'-3)
# --------------------------------------------------------------------------------------
def raw2outputs(raw, z_vals, rays_d, noise=None, white_bkgd=False, dtype=f32):
    """Returns dict(rgb_map, disp_map, acc_map, weights, depth_map, alpha).  `noise` is the
    already-scaled additive noise on raw[...,3] ([N,S]) or None."""
    raw = np.asarray(raw, dtype=dtype)
    z = np.asarray(z_vals, dtype=dtype)
    rays_d = np.asarray(rays_d, dtype=dtype)
    dists = (z[:, 1:] - z[:, :-1]).astype(dtype)                              # :367
    dists = np.concatenate([dists, np.full_like(dists[:, :1], 1e10)], -1)     # :368
    norm = np.sqrt((rays_d * rays_d).astype(dtype).sum(-1, dtype=dtype)).astype(dtype)[:, None]
    dists = (dists * norm).astype(dtype)                                      # :370
    rgb = (1.0 / (1.0 + np.exp(-raw[..., :3].astype(np.float64)))).astype(dtype)   # :372 sigmoid
    sig = raw[..., 3] if noise is None else (raw[..., 3] + np.asarray(noise, dtype=dtype)).astype(dtype)
    with np.errstate(over="ignore", invalid="ignore"):
        alpha = (1.0 - np.exp(-(np.maximum(sig, 0) * dists).astype(dtype))).astype(dtype)   # :365,:383
    q = ((1.0 - alpha).astype(dtype) + dtype(1e-10)).astype(dtype)
    T = np.cumprod(np.concatenate([np.ones_like(q[:, :1]), q], -1).astype(np.float64), -1)[:, :-1].astype(dtype)
    weights = (alpha * T).astype(dtype)                                       # :385
    rgb_map = (weights[..., None] * rgb).sum(-2, dtype=dtype)                 # :389
    depth_map = (weights * z).sum(-1, dtype=dtype)                            # :391
    acc_map = weights.sum(-1, dtype=dtype)                                    # :394
    with np.errstate(divide="ignore", invalid="ignore"):
        ratio = (depth_map / acc_map).astype(dtype)
        # torch.max(1e-10, x) propagates NaN (0/0 when every sigma<=0): keep it
        mx = np.where(np.isnan(ratio), ratio, np.maximum(dtype(1e-10), ratio))
        disp_map = (1.0 / mx).astype(dtype)                                   # :392
    if white_bkgd:
        rgb_map = (rgb_map + (1.0 - acc_map[:, None])).astype(dtype)          # :397
    return {"rgb_map": rgb_map, "disp_map": disp_map, "acc_map": acc_map,
            "weights": weights, "depth_map": depth_map, "alpha": alpha}


def raw2outputs_backward(raw, z_vals, rays_d, noise, white_bkgd,
                         g_rgb, g_disp, g_acc, g_depth, g_weights=None,
                         detach_weights=False, dtype=np.float64):
    """d raw [N,S,4] for upstream grads on (rgb_map, disp_map, acc_map, depth_map, weights).
    Closed form of SURVEY.md §8a'-3 (one forward product scan + one reverse sum scan)."""
    raw = np.asarray(raw, dtype=dtype)
    z = np.asarray(z_vals, dtype=dtype)
    rays_d = np.asarray(rays_d, dtype=dtype)
    N, S = z.shape
    dists = np.concatenate([z[:, 1:] - z[:, :-1], np.full((N, 1), 1e10, dtype=dtype)], -1)
    delta = dists * np.sqrt((rays_d * rays_d).sum(-1))[:, None]
    sig = raw[..., 3] + (0 if noise is None else np.asarray(noise, dtype=dtype))
    with np.errstate(over="ignore", invalid="ignore"):
        e = np.exp(-np.maximum(sig, 0) * delta)
    alpha = 1.0 - e
    q = (1.0 - alpha) + 1e-10
    T = np.cumprod(np.concatenate([np.ones((N, 1), dtype=dtype), q], -1), -1)[:, :-1]
    w = alpha * T
    c = 1.0 / (1.0 + np.exp(-raw[..., :3]))
    Dm = (w * z).sum(-1)
    A = w.sum(-1)
    with np.errstate(divide="ignore", invalid="ignore"):
        r = Dm / A
        live = ~(r <= 1e-10)      # torch.max(1e-10, r) backward: r==NaN keeps the grad path (-> NaN), like the reference
        gD = np.asarray(g_depth, dtype=dtype) + np.where(live, -np.asarray(g_disp, dtype=dtype) * A / (Dm * Dm), 0.0)
        gA = np.asarray(g_acc, dtype=dtype) + np.where(live, np.asarray(g_disp, dtype=dtype) / Dm, 0.0)
    g_rgb = np.asarray(g_rgb, dtype=dtype)
    if white_bkgd:
        gA = gA - g_rgb.sum(-1)
    G = z * gD[:, None] + gA[:, None]
    if not detach_weights:
        G = G + (c * g_rgb[:, None, :]).sum(-1)
    if g_weights is not None:
        G = G + np.asarray(g_weights, dtype=dtype)
    Gw = G * w
    suffix = np.cumsum(Gw[:, ::-1], -1)[:, ::-1] - Gw         # sum_{k>i} G_k w_k
    d_alpha = G * T - suffix / q
    with np.errstate(invalid="ignore", over="ignore"):
        d_sig = np.where(sig > 0, d_alpha * delta * e, 0.0)
        d_sig = np.where((sig > 0) & (e == 0), 0.0, d_sig)     # inf*0 (last interval) -> 0, as autograd's exp(-x)*x path gives
    d_rgb = w[..., None] * g_rgb[:, None, :] * c * (1.0 - c)
    return np.concatenate([d_rgb, d_sig[..., None]], -1)


# --------------------------------------------------------------------------------------
# a12/a13: depth -> xyz -> least-squares plane normal   (run.py:1909-1940)
# --------------------------------------------------------------------------------------
def _box_sum(img, k):
    """Sum over a k x k window with zero padding (== unfold(k, padding=k//2), run.py:1928)."""
    r = k // 2
    H, W = img.shape[:2]
    pad = np.zeros((H + 2 * r + 1, W + 2 * r + 1) + img.shape[2:], dtype=np.float64)
    pad[r + 1:r + 1 + H, r + 1:r + 1 + W] = img
    ii = pad.cumsum(0).cumsum(1)
    return ii[k:k + H, k:k + W] - ii[:H, k:k + W] - ii[k:k + H, :W] + ii[:H, :W]


def depth2xyz(depth, fx, fy, cx, cy):
    """run.py:1909-1922."""
    H, W = depth.shape
    hh, ww = np.mgrid[0:H, 0:W]
    z = np.asarray(depth, dtype=np.float64)
    x = (ww - cx) * z / fx
    y = (hh - cy) * z / fy
    return np.stack([x, y, z], -1)


def normal_from_depth(depth, fx, fy, cx, cy, k=31):
    """depth2normal_geo(depth2xyz_torch(depth)) (run.py:1924-1940): per pixel
    n = (A^T A)^-1 A^T 1 over the zero-padded k x k window == M^-1 s with
    M = sum a a^T, s = sum a over in-bounds pixels.  Returns [3,H,W] (un-normalised),
    computed in float64."""
    a = depth2xyz(depth, fx, fy, cx, cy)
    H, W, _ = a.shape
    s = _box_sum(a, k)
    outer = a[..., :, None] * a[..., None, :]
    M = _box_sum(outer.reshape(H, W, 9), k).reshape(H, W, 3, 3)
    n = np.linalg.solve(M, s[..., None])[..., 0]
    return np.transpose(n, (2, 0, 1))


def normal_from_depth_backward(depth, fx, fy, cx, cy, g_normal, k=31):
    """d depth [H,W] for upstream g_normal [3,H,W] (SURVEY.md §8a'-4)."""
    a = depth2xyz(depth, fx, fy, cx, cy)
    H, W, _ = a.shape
    s = _box_sum(a, k)
    outer = a[..., :, None] * a[..., None, :]
    M = _box_sum(outer.reshape(H, W, 9), k).reshape(H, W, 3, 3)
    n = np.linalg.solve(M, s[..., None])[..., 0]
    g = np.transpose(np.asarray(g_normal, dtype=np.float64), (1, 2, 0))
    qv = np.linalg.solve(M, g[..., None])[..., 0]           # M symmetric
    Q = _box_sum(qv, k)
    qn = qv[..., :, None] * n[..., None, :]
    Sym = _box_sum((qn + np.transpose(qn, (0, 1, 3, 2))).reshape(H, W, 9), k).reshape(H, W, 3, 3)
    da = Q - np.einsum("hwij,hwj->hwi", Sym, a)
    hh, ww = np.mgrid[0:H, 0:W]
    return da[..., 0] * (ww - cx) / fx + da[..., 1] * (hh - cy) / fy + da[..., 2]


# --------------------------------------------------------------------------------------
# a2: render_rays   (run.py:1703-1847) — the composed path used as the CPU baseline
# --------------------------------------------------------------------------------------
def render_rays(rays, p_coarse, p_fine, t_vals, t_rand=None, u=None, noise0=None, noise1=None,
                lindisp=False, white_bkgd=False, N_importance=64, dtype=f32):
    """rays [N,11] = (o, d, near, far, viewdir).  Randoms are inputs (host-generated in the
    reference's draw order, SURVEY.md §7 'RNG parity').  u defaults to the deterministic
    linspace row (perturb == 0)."""
    rays = np.asarray(rays, dtype=f32)
    viewdirs = rays[:, -3:]
    z = sample_coarse(rays, t_vals, t_rand, lindisp)
    raw0 = run_network(p_coarse, points(rays, z), viewdirs, dtype=dtype)
    c0 = raw2outputs(raw0, z, rays[:, 3:6], noise0, white_bkgd, dtype=dtype)
    if u is None:
        u = linspace_f32(0.0, 1.0, N_importance)
    fs = fine_samples(z, c0["weights"], u)
    zf = fs["z_merged"]
    raw1 = run_network(p_fine, points(rays, zf), viewdirs, dtype=dtype)
    c1 = raw2outputs(raw1, zf, rays[:, 3:6], noise1, white_bkgd, dtype=dtype)
    ret = {"rgb_map": c1["rgb_map"], "disp_map": c1["disp_map"], "acc_map": c1["acc_map"],
           "depth_map": c1["depth_map"], "weights": c1["weights"], "z_vals": zf, "raw": raw1,
           "alpha": c1["alpha"], "alpha0": c0["alpha"],
           "rgb0": c0["rgb_map"], "disp0": c0["disp_map"], "acc0": c0["acc_map"],
           "z_std": fs["z_std"], "z_coarse": z, "raw0": raw0, "weights0": c0["weights"],
           "z_samples": fs["z_samples"], "inds": fs["inds"], "depth0": c0["depth_map"]}
    return ret


def get_rays(H, W, focal, c2w):
    """run_nerf_helpers.py:249-260 (pinhole rays, float32)."""
    i, j = np.meshgrid(np.arange(W, dtype=f32), np.arange(H, dtype=f32), indexing="xy")
    dirs = np.stack([(i - f32(W * .5)) / f32(focal), -(j - f32(H * .5)) / f32(focal), -np.ones_like(i)], -1).astype(f32)
    c2w = np.asarray(c2w, dtype=f32)
    rays_d = (dirs[..., None, :] * c2w[:3, :3]).astype(f32).sum(-1, dtype=f32)
    rays_o = np.broadcast_to(c2w[:3, -1], rays_d.shape).astype(f32)
    return rays_o, rays_d


def ndc_rays(H, W, focal, near, rays_o, rays_d):
    """run_nerf_helpers.py:283-300.  Python-float scalars are formed in double and rounded to fp32 where they meet a
    tensor; `c / tensor` is reciprocal(tensor) * c (Tensor.__rtruediv__); every tensor op rounds to fp32."""
    rays_o = np.asarray(rays_o, dtype=f32)
    rays_d = np.asarray(rays_d, dtype=f32)
    t = (-(f32(near) + rays_o[..., 2]) / rays_d[..., 2]).astype(f32)
    rays_o = (rays_o + (t[..., None] * rays_d).astype(f32)).astype(f32)
    sx = f32(-1. / (W / (2. * focal)))
    sy = f32(-1. / (H / (2. * focal)))
    rz = (f32(1.) / rays_o[..., 2]).astype(f32)
    o0 = ((sx * rays_o[..., 0]).astype(f32) / rays_o[..., 2]).astype(f32)
    o1 = ((sy * rays_o[..., 1]).astype(f32) / rays_o[..., 2]).astype(f32)
    o2 = (f32(1.) + (rz * f32(2. * near)).astype(f32)).astype(f32)
    d0 = (sx * ((rays_d[..., 0] / rays_d[..., 2]).astype(f32) - (rays_o[..., 0] / rays_o[..., 2]).astype(f32)).astype(f32)).astype(f32)
    d1 = (sy * ((rays_d[..., 1] / rays_d[..., 2]).astype(f32) - (rays_o[..., 1] / rays_o[..., 2]).astype(f32)).astype(f32)).astype(f32)
    d2 = (rz * f32(-2. * near)).astype(f32)
    return np.stack([o0, o1, o2], -1), np.stack([d0, d1, d2], -1)


def _norm3(v):
    """torch.norm(v, dim=-1) for 3-vectors on CPU: sqrt(fma(z, z, fma(y, y, x*x))) — evaluated in double and rounded once per
    step, which equals the fused fp32 operations (a product of two fp32 is exact in double)."""
    x, y, z = [np.asarray(v[..., k], dtype=np.float64) for k in range(3)]
    a = (x * x).astype(f32).astype(np.float64)
    a = (y * y + a).astype(f32).astype(np.float64)
    a = (z * z + a).astype(f32)
    return np.sqrt(a).astype(f32)


def make_ray_batch(rays_o, rays_d, near, far, use_viewdirs=True, view_d=None, ndc=False, H=0, W=0, focal=1., ndc_near=1.):
    """render(): run.py:1176-1207 -> [N, 8 | 11] (o, d, near, far[, viewdir]); view_d = directions the view vectors come from
    when they differ from rays_d (c2w_staticcam)."""
    rays_o = np.asarray(rays_o, dtype=f32).reshape(-1, 3)
    rays_d = np.asarray(rays_d, dtype=f32).reshape(-1, 3)
    vsrc = rays_d if view_d is None else np.asarray(view_d, dtype=f32).reshape(-1, 3)
    viewdirs = (vsrc / _norm3(vsrc)[:, None]).astype(f32)
    if ndc:
        rays_o, rays_d = ndc_rays(H, W, focal, ndc_near, rays_o, rays_d)
    n = np.full_like(rays_d[:, :1], near)
    f = np.full_like(rays_d[:, :1], far)
    return np.concatenate([rays_o, rays_d, n, f] + ([viewdirs] if use_viewdirs else []), -1).astype(f32)


# --------------------------------------------------------------------------------------
# Model of the CUDA path's mixed precision (bf16 tensor-core operands, fp32/fp64 accumulate).
# Not a restatement of the reference: it answers "is the kernel computing what it is specified
# to compute" separately from "how far is bf16 from the reference's fp32" (ReLU-mask flips of
# ~0.5% of units dominate the latter for gradients).
# --------------------------------------------------------------------------------------
def bf16_round(x):
    """round-to-nearest-even float32 -> bfloat16 -> float64 (numpy bit arithmetic)."""
    a = np.ascontiguousarray(x, dtype=np.float32).view(np.uint32).astype(np.uint64)
    a = (a + 0x7FFF + ((a >> 16) & 1)) & 0xFFFF0000
    return a.astype(np.uint32).view(np.float32).reshape(np.shape(x)).astype(np.float64)


def nerf_forward_backward_bf16sim(p, pts, viewdirs, d_out=None, multires=10, multires_views=4, keep=False):
    """Forward (and, with d_out, backward) of the NeRF MLP with every tensor-core operand rounded to
    bf16 exactly where the kernels round: MMA weights, PE inputs, each layer's activation, each dZ.
    The alpha / rgb heads run on fp32 activations with fp32 weights, as in mlp_forward.cu.
    keep=True appends a dict of the intermediates: pe, vpe, ins / pre / h (input, pre-activation and bf16 output of each
    pts_linears layer), feat, pre_v, hidden (bf16), and with d_out d_hidden_pre, d_feat and dz (dZ of each pts_linears layer)."""
    W = {k: (bf16_round(v) if (k.endswith("weight") and not k.startswith(("alpha", "rgb"))) else v.astype(np.float64))
         for k, v in p.items()}
    pe = bf16_round(embed(pts, multires))
    vpe = bf16_round(embed(viewdirs, multires_views))
    h = pe
    ins, pre, outs = [], [], []
    h8_f = None
    for i in range(8):
        ins.append(h)
        z = h @ W["pts_linears.%d.weight" % i].T + W["pts_linears.%d.bias" % i]
        pre.append(z)
        hf = np.maximum(z, 0)
        h = bf16_round(hf)
        outs.append(h)
        if i == 7:
            h8_f = hf
        if i == 4:
            h = np.concatenate([pe, h], -1)
    h8 = h
    alpha = h8_f @ W["alpha_linear.weight"].T + W["alpha_linear.bias"]
    feat = bf16_round(h8 @ W["feature_linear.weight"].T + W["feature_linear.bias"])
    hv_in = np.concatenate([feat, vpe], -1)
    pre_v = hv_in @ W["views_linears.0.weight"].T + W["views_linears.0.bias"]
    hv_f = np.maximum(pre_v, 0)
    rgb = hv_f @ W["rgb_linear.weight"].T + W["rgb_linear.bias"]
    out = np.concatenate([rgb, alpha], -1)
    saved = dict(pe=pe, vpe=vpe, ins=ins, pre=pre, h=outs, feat=feat, pre_v=pre_v, hidden=bf16_round(hv_f))
    if d_out is None:
        return (out, saved) if keep else out
    g = {}
    d_out = np.asarray(d_out, dtype=np.float64)
    d_rgb, d_alpha = d_out[:, :3], d_out[:, 3:4]
    hv = bf16_round(hv_f)
    g["rgb_linear.weight"] = d_rgb.T @ hv
    g["rgb_linear.bias"] = d_rgb.sum(0)
    g["alpha_linear.weight"] = d_alpha.T @ h8
    g["alpha_linear.bias"] = d_alpha.sum(0)
    d_pre_v = bf16_round((d_rgb @ W["rgb_linear.weight"]) * (pre_v > 0))
    g["views_linears.0.weight"] = d_pre_v.T @ hv_in
    g["views_linears.0.bias"] = d_pre_v.sum(0)
    d_feat = bf16_round((d_pre_v @ W["views_linears.0.weight"])[:, :256])
    g["feature_linear.weight"] = d_feat.T @ h8
    g["feature_linear.bias"] = d_feat.sum(0)
    d_h = d_feat @ W["feature_linear.weight"] + d_alpha @ W["alpha_linear.weight"]
    dz = [None] * 8
    for i in reversed(range(8)):
        if i == 4:
            d_h = d_h[:, 63:]
        d_pre = dz[i] = bf16_round(d_h * (pre[i] > 0))
        g["pts_linears.%d.weight" % i] = d_pre.T @ ins[i]
        g["pts_linears.%d.bias" % i] = d_pre.sum(0)
        d_h = d_pre @ W["pts_linears.%d.weight" % i]
    if keep:
        saved.update(d_hidden_pre=d_pre_v, d_feat=d_feat, dz=dz)
        return out, g, saved
    return out, g


# --------------------------------------------------------------------------------------
# One training step of the path (render_rays forward + backward of an MSE loss), used as the CPU
# baseline by bench.py (`cpu_baseline` / `--impl reference`, kind "port") and by the e2e tests.
# --------------------------------------------------------------------------------------
def train_step(rays, p_coarse, p_fine, t_vals, t_rand, u, noise0, noise1, target_rgb, lindisp=True,
               white_bkgd=True, dtype=f32):
    """loss = mse(rgb, target) + mse(rgb0, target) (run.py:1000-1027 without the SDS / depth terms);
    returns (loss, grads_coarse, grads_fine).  Follows autograd of the reference: z_samples detached."""
    rays = np.asarray(rays, dtype=f32)
    N = rays.shape[0]
    viewdirs = rays[:, -3:]
    z0 = sample_coarse(rays, t_vals, t_rand, lindisp)
    raw0, saved0 = run_network(p_coarse, points(rays, z0), viewdirs, keep=True, dtype=dtype)
    c0 = raw2outputs(raw0, z0, rays[:, 3:6], noise0, white_bkgd, dtype=dtype)
    fs = fine_samples(z0, c0["weights"], u)
    z1 = fs["z_merged"]
    raw1, saved1 = run_network(p_fine, points(rays, z1), viewdirs, keep=True, dtype=dtype)
    c1 = raw2outputs(raw1, z1, rays[:, 3:6], noise1, white_bkgd, dtype=dtype)
    target = np.asarray(target_rgb, dtype=np.float64)
    d1 = c1["rgb_map"].astype(np.float64) - target
    d0 = c0["rgb_map"].astype(np.float64) - target
    loss = float((d1 ** 2).mean() + (d0 ** 2).mean())
    g_rgb1 = 2.0 * d1 / d1.size
    g_rgb0 = 2.0 * d0 / d0.size
    zeros = np.zeros(N)
    d_raw1 = raw2outputs_backward(raw1, z1, rays[:, 3:6], noise1, white_bkgd, g_rgb1, zeros, zeros, zeros, dtype=np.float64)
    d_raw0 = raw2outputs_backward(raw0, z0, rays[:, 3:6], noise0, white_bkgd, g_rgb0, zeros, zeros, zeros, dtype=np.float64)
    g1 = nerf_backward(p_fine, saved1, d_raw1.reshape(-1, 4).astype(dtype), dtype=dtype)
    g0 = nerf_backward(p_coarse, saved0, d_raw0.reshape(-1, 4).astype(dtype), dtype=dtype)
    return loss, g0, g1


def blas_threads():
    """Number of threads numpy's BLAS uses (what `cores` means in bench.py's cpu_baseline)."""
    try:
        from threadpoolctl import threadpool_info
        n = [i.get("num_threads", 1) for i in threadpool_info() if i.get("user_api") == "blas"]
        if n:
            return int(max(n))
    except Exception:
        pass
    import os
    return os.cpu_count() or 1
