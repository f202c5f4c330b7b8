"""GPU suite: fused PE + NeRF MLP (tcgen05) against the reference's NeRF.forward (golden) and the oracle."""
import numpy as np
import pytest
import torch

import mlp_ref64 as ref
from oracle import nerf_oracle as orc

pytestmark = pytest.mark.gpu

# bf16 operands / fp32 accumulate.  Stated tolerances (random-init network, SURVEY.md §8c):
RAW_ATOL = 2e-2        # max-abs on raw (rgb logits, sigma)
RGB_ATOL = 2e-3        # max-abs on composited rgb
DEPTH_RTOL = 1e-2      # relative on composited depth


@pytest.fixture(scope="module")
def ops():
    from mvip_nerf_b200 import ops as o
    return o


def cu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def pack(ops, p):
    return ops.mlp_pack([cu(p[n]) for n in ops.PARAM_ORDER])


def test_pack_layout_roundtrip(ops):
    p = orc.init_params(3)
    blob = pack(ops, p).cpu().numpy()
    w = blob[:34 * 32768 + 5 * 16384].view(np.uint16)
    # chunk 1 = pts_linears.1 columns 0..63: element (n, k) at byte (n>>3)*1024 + (n&7)*128 + ((k>>3 ^ n&7)<<4) + (k&7)*2
    W1 = torch.from_numpy(p["pts_linears.1.weight"]).bfloat16().view(torch.int16).numpy().view(np.uint16)
    for n, k in [(0, 0), (5, 9), (200, 63), (255, 17)]:
        off = 32768 + (n >> 3) * 1024 + (n & 7) * 128 + (((k >> 3) ^ (n & 7)) << 4) + (k & 7) * 2
        assert w[off // 2] == W1[n, k]
    small = blob[34 * 32768 + 5 * 16384 + 34 * 32768:].view(np.float32)
    assert np.array_equal(small[:256], p["pts_linears.0.bias"])
    assert np.array_equal(small[2432:2688], p["alpha_linear.weight"][0])
    assert np.array_equal(small[2692:2692 + 384], p["rgb_linear.weight"].ravel())


def test_mlp_forward_points_vs_reference(ops, golden):
    fx = golden("nerf_mlp")
    p = orc.init_params(int(fx["param_seed"]))
    emb = cu(fx["embedded"])
    # the drop-in NeRF.forward path: raw pts / viewdirs are columns 0:3 and 63:66 of the embedded input
    raw = ops.mlp_forward(pack(ops, p), pts=emb[:, 0:3], dirs=emb[:, 63:66])
    err = np.abs(raw.cpu().numpy() - fx["out"]).max()
    assert err < RAW_ATOL, err


@pytest.mark.parametrize("P", [1, 127, 128, 129, 300, 5000])
def test_mlp_forward_ragged_sizes_vs_oracle(ops, P):
    rng = np.random.RandomState(P)
    p = orc.init_params(11)
    pts = ((rng.rand(P, 3) * 2 - 1) * 6).astype(np.float32)
    vd = rng.randn(P, 3).astype(np.float32)
    vd /= np.linalg.norm(vd, axis=-1, keepdims=True)
    want = orc.nerf_forward(p, np.concatenate([orc.embed(pts, 10), orc.embed(vd, 4)], -1))
    raw = ops.mlp_forward(pack(ops, p), pts=cu(pts), dirs=cu(vd))
    assert raw.shape == (P, 4)
    err = np.abs(raw.cpu().numpy() - want).max()
    assert err < RAW_ATOL, err


def test_mlp_forward_rays_mode_and_stash_do_not_change_result(ops):
    rng = np.random.RandomState(5)
    N, S = 96, 64
    p = orc.init_params(12)
    ro, rd = orc.get_rays(756, 1008, 767.2935, np.eye(4, dtype=np.float32)[:3, :4])
    idx = rng.permutation(756 * 1008)[:N]
    rays = orc.make_ray_batch(ro.reshape(-1, 3)[idx], rd.reshape(-1, 3)[idx], 1.2, 7.7369)
    z = orc.sample_coarse(rays, orc.linspace_f32(0, 1, S), rng.rand(N, S).astype(np.float32), True)
    want = orc.run_network(p, orc.points(rays, z), rays[:, -3:])
    blob = pack(ops, p)
    raw = ops.mlp_forward(blob, rays=cu(rays), z_vals=cu(z))
    err = np.abs(raw.view(N, S, 4).cpu().numpy() - want).max()
    assert err < RAW_ATOL, err
    raw2, stash = ops.mlp_forward(blob, rays=cu(rays), z_vals=cu(z), want_stash=True)
    assert torch.equal(raw, raw2)
    # stash chunk 0 of tile 0 is the PE tile image: row 0, first 3 bf16 = the point itself
    pe0 = stash[:6].cpu().view(torch.bfloat16).float().numpy()
    np.testing.assert_allclose(pe0, orc.points(rays, z)[0, 0], rtol=1e-2)


def test_mlp_forward_is_deterministic_and_tile_independent(ops):
    # size-independent property at cfg-2 size: a point's output does not depend on its tile / neighbours
    rng = np.random.RandomState(9)
    P = 4096 * 64
    p = orc.init_params(13)
    pts = ((rng.rand(P, 3) * 2 - 1) * 4).astype(np.float32)
    vd = rng.randn(P, 3).astype(np.float32)
    blob = pack(ops, p)
    a = ops.mlp_forward(blob, pts=cu(pts), dirs=cu(vd))
    b = ops.mlp_forward(blob, pts=cu(pts), dirs=cu(vd))
    assert torch.equal(a, b)
    perm = torch.randperm(P, device="cuda")
    c = ops.mlp_forward(blob, pts=cu(pts)[perm].contiguous(), dirs=cu(vd)[perm].contiguous())
    assert torch.equal(a[perm], c)
    sub = rng.permutation(P)[:2048]
    want = orc.nerf_forward(p, np.concatenate([orc.embed(pts[sub], 10), orc.embed(vd[sub], 4)], -1))
    assert np.abs(a.cpu().numpy()[sub] - want).max() < RAW_ATOL


# Gradients.  Two checks with different meanings:
#  (a) teacher-forced: decode the kernel's own activation stash (bf16 tile images + ReLU bit masks) and recompute
#      the backward in float64 with the same operand roundings -> every kernel of the backward (dgrad chain,
#      wgrad, heads, reduce) must agree to GRAD_TF_RTOL of each tensor's max-abs entry;
#  (b) against the reference's fp32 autograd: bf16 flips ~0.5% of the ReLU masks, which for a random upstream
#      gradient is a ~5-10% L2 effect (reproduced on CPU by oracle.nerf_forward_backward_bf16sim) -> stated
#      tolerance: cosine >= 0.99 and max-abs error <= 25% of the tensor's max-abs entry; heads <= 1%.
GRAD_TF_RTOL = 5e-3
GRAD_REF_COS = 0.99
GRAD_REF_RTOL = 0.25

def teacher_forced_grads(p, stash, P, d_out):
    """float64 backward from the decoded stash, rounding dZ to bf16 where the dgrad chain does (mlp_ref64)"""
    g = ref.teacher_forced_grads(p, stash, P, torch.as_tensor(np.asarray(d_out, dtype=np.float32)))
    return {n: v.cpu().numpy() for n, v in g.items()}


def _check_grads(ops, got, want_by_name, P, teacher_forced):
    for g, name in zip(got, ops.PARAM_ORDER):
        ref = np.asarray(want_by_name[name], dtype=np.float64).reshape(g.shape)
        a = g.cpu().numpy().astype(np.float64)
        scale = max(float(np.abs(ref).max()), 1e-12)
        err = float(np.abs(a - ref).max()) / scale
        if teacher_forced:
            assert err < GRAD_TF_RTOL, (name, err, P)
        else:
            head = name.startswith(("alpha", "rgb"))
            assert err < (1e-2 if head else GRAD_REF_RTOL), (name, err, P)
            if a.size > 8 and P >= 64:
                cos = float((a * ref).sum() / np.sqrt((a * a).sum() * (ref * ref).sum()))
                assert cos > GRAD_REF_COS, (name, cos, P)


def test_mlp_backward_vs_reference_autograd(ops, golden):
    fx = golden("nerf_mlp")
    p = orc.init_params(int(fx["param_seed"]))
    blob = pack(ops, p)
    emb = cu(fx["embedded"])
    P = emb.shape[0]
    raw, stash = ops.mlp_forward(blob, pts=emb[:, 0:3], dirs=emb[:, 63:66], want_stash=True)
    grads = ops.mlp_backward(blob, cu(fx["d_out"]), stash)
    _check_grads(ops, grads, {n: fx["grad." + n] for n in ops.PARAM_ORDER}, P, teacher_forced=False)
    _check_grads(ops, grads, teacher_forced_grads(p, stash, P, fx["d_out"]), P, teacher_forced=True)
    # accumulate=True adds on top
    grads2 = ops.mlp_backward(blob, cu(fx["d_out"]), stash, grads=[g.clone() for g in grads], accumulate=True)
    for a, b in zip(grads, grads2):
        torch.testing.assert_close(b, 2 * a, rtol=1e-6, atol=1e-7)


def test_stash_matches_bf16_model(ops):
    # the stash is what the forward really computed: compare it with the CPU bf16 model, layer by layer
    rng = np.random.RandomState(77)
    P = 300
    p = orc.init_params(23)
    pts = ((rng.rand(P, 3) * 2 - 1) * 5).astype(np.float32)
    vd = rng.randn(P, 3).astype(np.float32)
    raw, stash = ops.mlp_forward(pack(ops, p), pts=cu(pts), dirs=cu(vd), want_stash=True)
    st = ref.decode_stash(stash, P, range(ref.num_tiles(P)))
    st = {k: [x[:P].cpu().numpy() for x in v] if isinstance(v, list) else v[:P].cpu().numpy() for k, v in st.items() if k != "finite"}
    np.testing.assert_allclose(st["pe"][:, :63], orc.bf16_round(orc.embed(pts, 10)), atol=8e-3)   # 1 bf16 ulp at |x|<=1... sin/cos
    np.testing.assert_allclose(st["vpe"][:, :27], orc.bf16_round(orc.embed(vd, 4)), atol=2e-2)
    assert np.all(st["pe"][:, 63] == 0) and np.all(st["vpe"][:, 27:] == 0)
    for l in range(8):
        assert np.array_equal(st["mask"][l], st["h"][l] > 0)         # bit masks == sign of the stored activations
    assert np.array_equal(st["mask"][8], st["hidden"] > 0)
    out_m = orc.nerf_forward_backward_bf16sim(p, pts, vd)
    assert np.abs(raw.cpu().numpy() - out_m).max() < 2e-3


@pytest.mark.parametrize("P", [1, 129, 1000, 20000])
def test_mlp_backward_ragged_sizes_vs_oracle(ops, P):
    rng = np.random.RandomState(100 + P)
    p = orc.init_params(21)
    pts = ((rng.rand(P, 3) * 2 - 1) * 5).astype(np.float32)
    vd = rng.randn(P, 3).astype(np.float32)
    vd /= np.linalg.norm(vd, axis=-1, keepdims=True)
    d_out = rng.randn(P, 4).astype(np.float32)
    blob = pack(ops, p)
    raw, stash = ops.mlp_forward(blob, pts=cu(pts), dirs=cu(vd), want_stash=True)
    grads = ops.mlp_backward(blob, cu(d_out), stash)
    _check_grads(ops, grads, teacher_forced_grads(p, stash, P, d_out), P, teacher_forced=True)
    if P >= 1000:
        x = np.concatenate([orc.embed(pts, 10), orc.embed(vd, 4)], -1)
        _, saved = orc.nerf_forward(p, x, keep=True, dtype=np.float64)
        _check_grads(ops, grads, orc.nerf_backward(p, saved, d_out, dtype=np.float64), P, teacher_forced=False)


def test_mlp_backward_is_linear_and_deterministic_at_full_size(ops):
    # cfg-2 coarse-pass size (4096 rays x 64): grads are linear in d_raw and bitwise reproducible
    rng = np.random.RandomState(3)
    P = 4096 * 64
    p = orc.init_params(22)
    blob = pack(ops, p)
    pts = cu(((rng.rand(P, 3) * 2 - 1) * 4).astype(np.float32))
    vd = cu(rng.randn(P, 3).astype(np.float32))
    d1 = cu(rng.randn(P, 4).astype(np.float32))
    raw, stash = ops.mlp_forward(blob, pts=pts, dirs=vd, want_stash=True)
    g1 = ops.mlp_backward(blob, d1, stash)
    g1b = ops.mlp_backward(blob, d1, stash)
    for a, b in zip(g1, g1b):
        assert torch.equal(a, b)
    g2 = ops.mlp_backward(blob, 2 * d1, stash)
    for a, b, name in zip(g1, g2, ops.PARAM_ORDER):
        scale = float(a.abs().max())
        assert float((b - 2 * a).abs().max()) <= 2e-2 * scale, name     # bf16 rounding of dZ is not exactly linear
    # bias grad of rgb_linear is exactly the column sum of d_raw[:, :3]
    torch.testing.assert_close(g1[23], d1[:, :3].sum(0), rtol=1e-4, atol=1e-2)
    torch.testing.assert_close(g1[21], d1[:, 3:].sum(0), rtol=1e-4, atol=1e-2)




@pytest.mark.gpu
def test_fused_backward_is_deterministic_and_never_reads_stale_dz():
    """The fused backward hands dZ from the chain to the wgrad role through per-(tile, group) flags.  A consumer that ran ahead of
    its producer would read whatever the workspace held before: the workspace is therefore POISONED (NaN bit patterns) before
    each run - any premature read shows up as NaN / a different bit pattern - and three runs must agree bit for bit."""
    import ctypes
    from mvip_nerf_b200 import _lib, ops
    dev = "cuda"
    p = orc.init_params(7)
    blob = ops.mlp_pack([torch.from_numpy(p[n]).to(dev) for n in ops.PARAM_ORDER])
    g = torch.Generator(device=dev).manual_seed(11)
    P = 128 * 148 * 6 + 53
    pts = torch.rand(P, 3, device=dev, generator=g) * 4 - 2
    dirs = torch.nn.functional.normalize(torch.randn(P, 3, device=dev, generator=g), dim=-1)
    raw, stash = ops.mlp_forward(blob, pts=pts, dirs=dirs, want_stash=True)
    d = torch.randn(P, 4, device=dev, generator=g)
    lib = _lib.load()
    ws = ops._aligned_bytes(lib.mvip_mlp_backward_workspace_bytes(P), dev)
    outs = []
    for rep in range(3):
        ws.fill_(0xFF)                                  # bf16 0xFFFF = NaN, flags != 0 are reset by the library itself
        flat = torch.full((595844,), float("nan"), device=dev)
        grads, off = [], 0
        for shp in ops.PARAM_SHAPES:
            n = int(torch.Size(shp).numel())
            grads.append(flat[off:off + n].view(shp)); off += n
        arr = (ctypes.c_void_p * 24)(*[x.data_ptr() for x in grads])
        rc = lib.mvip_mlp_backward(ops._ptr(blob), ops._ptr(d), P, ops._ptr(stash), ops._ptr(ws), arr, 0, ops._stream())
        _lib.check(rc, "mvip_mlp_backward")
        torch.cuda.synchronize()
        outs.append(flat.clone())
    assert torch.isfinite(outs[0]).all()
    assert torch.equal(outs[0], outs[1]) and torch.equal(outs[0], outs[2])


@pytest.mark.gpu
def test_fused_backward_does_not_depend_on_its_scheduling_knobs():
    """Stagger of the chain starts and the credit throttle only change WHEN things happen inside backward_fused_kernel: every
    wgrad pair still consumes its tiles in the same fixed order, so the gradients must be bit-identical for any setting
    (no stagger / no throttle, the defaults, an absurdly tight throttle that stalls every tile, a huge stagger)."""
    import ctypes
    from mvip_nerf_b200 import _lib, ops
    dev = "cuda"
    p = orc.init_params(9)
    blob = ops.mlp_pack([torch.from_numpy(p[n]).to(dev) for n in ops.PARAM_ORDER])
    g = torch.Generator(device=dev).manual_seed(13)
    P = 128 * 148 * 3 + 17
    pts = torch.rand(P, 3, device=dev, generator=g) * 4 - 2
    dirs = torch.nn.functional.normalize(torch.randn(P, 3, device=dev, generator=g), dim=-1)
    raw, stash = ops.mlp_forward(blob, pts=pts, dirs=dirs, want_stash=True)
    d = torch.randn(P, 4, device=dev, generator=g)
    lib = _lib.load()
    ws = ops._aligned_bytes(lib.mvip_mlp_backward_workspace_bytes(P), dev)
    outs = []
    try:
        for stagger, throttle in ((0, (500, 0, 0)), (-1, (500, 60000, 20)), (-1, (1, 20000, 0)), (5000, (50, 60000, 200))):
            lib.mvip_debug_set_bwd_stagger(stagger)
            lib.mvip_debug_set_bwd_throttle(*throttle)
            ws.fill_(0xFF)
            flat = torch.full((595844,), float("nan"), device=dev)
            grads, off = [], 0
            for shp in ops.PARAM_SHAPES:
                n = int(torch.Size(shp).numel())
                grads.append(flat[off:off + n].view(shp)); off += n
            arr = (ctypes.c_void_p * 24)(*[x.data_ptr() for x in grads])
            rc = lib.mvip_mlp_backward(ops._ptr(blob), ops._ptr(d), P, ops._ptr(stash), ops._ptr(ws), arr, 0, ops._stream())
            _lib.check(rc, "mvip_mlp_backward")
            torch.cuda.synchronize()
            outs.append(flat.clone())
    finally:
        lib.mvip_debug_set_bwd_stagger(-1)
        lib.mvip_debug_set_bwd_throttle(500, 60000, 20)
    assert torch.isfinite(outs[0]).all()
    for o in outs[1:]:
        assert torch.equal(outs[0], o)


def test_backward_after_a_repack_raises(ops):
    """The packed bf16 blob is shared and re-packed in place: a backward that runs after the parameters changed would use the
    NEW weights for dgrad (ADVICE r1).  NeRF records the pack generation at forward and refuses such a backward; an in-place
    parameter write followed by invalidate_packed() is picked up by the next forward."""
    from mvip_nerf_b200.run_nerf_helpers import NeRF
    torch.manual_seed(0)
    net = NeRF(D=8, W=256, input_ch=63, input_ch_views=27, output_ch=4, skips=[4], use_viewdirs=True).cuda()
    pts = torch.rand(300, 3, device="cuda") * 2 - 1
    dirs = torch.nn.functional.normalize(torch.randn(300, 3, device="cuda"), dim=-1)
    raw0 = net.query_points(pts, dirs)
    raw0.sum().backward()                                           # the normal order works
    assert all(p.grad is not None and torch.isfinite(p.grad).all() for p in net.parameters())
    raw1 = net.query_points(pts, dirs)
    with torch.no_grad():
        net.rgb_linear.bias.data.add_(0.25)                          # a raw .data write bumps no version counter ...
    net.invalidate_packed()                                          # ... so the contract is an explicit invalidation
    raw2 = net.query_points(pts, dirs)                               # re-packs: the new bias is visible
    assert float((raw2[:, :3] - raw1[:, :3] - 0.25).detach().abs().max()) < 1e-5
    with pytest.raises(RuntimeError, match="re-packed"):
        raw1.sum().backward()


def test_empty_batch_gives_zero_gradients(ops):
    """N_rays == 0 under grad (reachable from dist.shard_rows when rays < world): the backward launches nothing, so the 24
    gradients must come back as zeros, not as uninitialised memory that a sum-allreduce would spread (ADVICE r1)."""
    p = orc.init_params(2)
    blob = pack(ops, p)
    stash = torch.empty(0, dtype=torch.uint8, device="cuda")
    grads = ops.mlp_backward(blob, torch.empty(0, 4, device="cuda"), stash)
    assert len(grads) == 24 and all(float(g.abs().max()) == 0.0 for g in grads)
