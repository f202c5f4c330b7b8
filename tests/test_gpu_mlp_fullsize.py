"""GPU: EVERY tile of the fused MLP forward and backward against float64 (tests/mlp_ref64.py), at the sizes where the fused
backward's scheduling changes and at the sizes training runs.

backward_fused_kernel hands tile pairs to CTA pairs dynamically after the first wave, staggers the chain starts, throttles the
chains by the dZ units in flight and has wgrad pairs pick the published dZ units up out of L2.  A schedule that always skips,
double-counts or mis-assigns a tile is deterministic and linear in d_raw, so only value checks at these sizes can see it:

  * forward: each stored layer output is compared with bf16(relu(X W^T + b)) of its own DECODED input, the masks with the
    stored activations, raw with the float64 heads of the decoded rows, the PE images with float64 sin / cos;
  * backward: each dgrad-chain step is recomputed from the kernel's own previous dZ image (workspace offset 0), and all 24
    gradients from the decoded dZ and stash in float64: what is left is fp32 summation order, bounded elementwise relative to
    |dZ|^T |X|; the teacher-forced end-to-end bar of test_gpu_mlp stays as well;
  * every tile exactly once: for each tile and each of the ten weight gradients of the fused kernel, the kernel's error
    projected on that tile's float64 contribution must stay near 0 (a dropped tile gives -1, a double-counted one +1).
    The elementwise bar alone cannot promise that at training sizes: it grows with sqrt(tiles) (fp32 sum order), and one
    tile's share of an element falls below 10x the bar above ~5,000 tiles (measured on a B200: 22x at 2,048 tiles, 4x at
    6,144, < 1x for the 11-point last tile of the guidance chunk; recorded per size as tile_contribution_over_bar for the
    first, the last and one dynamically handed-out tile).

The stash is pre-filled with 0xFF (bf16 NaN), the workspace poisoned with 0xFF and the gradients with NaN; d_raw is a view of a
buffer whose 64 trailing rows are NaN, so a read past P shows up.  The measured maxima of every size are written as
mlp_fullsize.json by test_gpu_train_parity.record() (a B200 run is kept as profiles/r03_mlp_fullsize.json)."""
import ctypes
import time

import pytest
import torch

import mlp_ref64 as ref
import test_gpu_train_parity as parity
from oracle import nerf_oracle as orc

pytestmark = pytest.mark.gpu

GRAD_TF_RTOL = 5e-3          # end-to-end teacher-forced bar of test_gpu_mlp
N_GRADS = 595844
_RESULTS = {}


def record(name, obj):
    """one file for all sizes, rewritten after each"""
    _RESULTS[name] = obj
    parity.record("mlp_fullsize.json", _RESULTS)


# (id, number of points as a function of the number of CTA pairs n = SMs // 2, inputs).  On a B200 n = 74:
#   <= 2 n tiles = 18,944 points: one wave of tile pairs, no stagger;  2 n tiles + 1 point: dynamic hand-out and stagger on,
#   the last pair half empty;  > 4 n tiles = 37,888: the forward gives a cluster more than one quad of tiles;
#   cfg 2 coarse (4,096 rays x 64) / fine (x 192) in rays mode, a ragged size and the 8,192-ray guidance chunk (x 192) + 11:
#   the credit throttle engages, thousands of dZ units in flight.
CASES = [
    ("1", lambda n: 1, "pts"), ("127", lambda n: 127, "pts"), ("128", lambda n: 128, "pts"), ("129", lambda n: 129, "pts"),
    ("255", lambda n: 255, "pts"), ("256", lambda n: 256, "pts"), ("257", lambda n: 257, "pts"),
    ("n-1_tiles", lambda n: 128 * (n - 1), "pts"), ("n_tiles+1", lambda n: 128 * n + 1, "pts"),
    ("2n-1_tiles", lambda n: 128 * (2 * n - 1), "pts"),
    ("2n_tiles", lambda n: 128 * 2 * n, "pts"), ("2n_tiles+1", lambda n: 128 * 2 * n + 1, "pts"),
    ("2n+1_tiles", lambda n: 128 * (2 * n + 1), "pts"),
    ("4n_tiles", lambda n: 128 * 4 * n, "pts"), ("4n_tiles+1", lambda n: 128 * 4 * n + 1, "pts"),
    ("128077", lambda n: 128077, "pts"),
    ("cfg2_coarse_rays", lambda n: 4096 * 64, "coarse"),
    ("cfg2_fine_rays", lambda n: 4096 * 192, "fine"),
    ("786379", lambda n: 786379, "pts"),
    ("guidance_chunk+11", lambda n: 8192 * 192 + 11, "pts"),
    ("2^21+3", lambda n: 2 ** 21 + 3, "pts"),
]


def n_pairs():
    return torch.cuda.get_device_properties(0).multi_processor_count // 2


def inputs(ops, P, mode, blob, g):
    """-> (points struct args for ops._points_struct, fp32 points [P,3], fp32 viewdirs [P,3])"""
    dev = "cuda"
    if mode == "pts":
        pts = torch.rand(P, 3, device=dev, generator=g) * 8 - 4
        dirs = torch.nn.functional.normalize(torch.randn(P, 3, device=dev, generator=g), dim=-1)
        return dict(pts=pts, dirs=dirs), pts, dirs
    N = 4096
    ro = (torch.rand(N, 3, device=dev, generator=g) * 2 - 1) * 0.5
    rd = torch.randn(N, 3, device=dev, generator=g) * 0.3 + torch.tensor([0.0, 0.0, -1.0], device=dev)
    rays = ops.rays_pack(ro, rd, 2.0, 6.0)                                    # [N, 11], viewdirs at column 8
    t_vals = torch.from_numpy(orc.linspace_f32(0, 1, 64)).to(dev)
    z = ops.sample_coarse(rays, t_vals, torch.rand(N, 64, device=dev, generator=g), False)
    if mode == "fine":
        raw0 = ops.mlp_forward(blob, rays=rays, z_vals=z)
        w = ops.composite_forward(raw0.view(N, 64, 4), z, rays[:, 3:6])[3]
        z = ops.sample_fine(z, w, torch.rand(N, 128, device=dev, generator=g))["z_merged"]
    S = z.shape[1]
    assert N * S == P
    ray = torch.arange(P, device=dev) // S
    pts = rays[ray, 0:3] + rays[ray, 3:6] * z.reshape(-1, 1)                  # o + d z, no FMA: mlp_forward.cu
    return dict(rays=rays, z_vals=z), pts, rays[ray, 8:11]


def grad_views(flat):
    from mvip_nerf_b200 import ops
    out, off = [], 0
    for shp in ops.PARAM_SHAPES:
        n = int(torch.Size(shp).numel())
        out.append(flat[off:off + n].view(shp))
        off += n
    return out


def backward(lib, ops, blob, d_raw, P, stash, ws, flat, accumulate=0, phases=None):
    ws.fill_(0xFF)                                      # bf16 NaN; the flags are cleared by the library itself
    arr = (ctypes.c_void_p * 24)(*[x.data_ptr() for x in grad_views(flat)])
    from mvip_nerf_b200 import _lib
    if phases is None:
        _lib.check(lib.mvip_mlp_backward(ops._ptr(blob), ops._ptr(d_raw), P, ops._ptr(stash), ops._ptr(ws), arr, accumulate,
                                         ops._stream()), "mvip_mlp_backward")
    else:
        for bit in phases:
            _lib.check(lib.mvip_mlp_backward_phases(ops._ptr(blob), ops._ptr(d_raw), P, ops._ptr(stash), ops._ptr(ws), arr,
                                                    accumulate, bit, ops._stream()), "mvip_mlp_backward_phases")
    torch.cuda.synchronize()


def tile_contribution(stash, ws, d_raw, P, t, bars):
    """min over the 20 gradients of backward_fused_kernel (each is one scheduled work item) of
    max_e |contribution of tile t|_e / (|dZ|^T |X|)_e.  The alpha / rgb heads come from head_grads_kernel, which has no
    dynamic schedule."""
    tiles = range(t, t + 1)
    st = ref.decode_stash(stash, P, tiles)
    g, _ = ref.wgrad(st, ref.decode_dz(ws, P, tiles), ref.rows_of(d_raw, P, tiles))
    return min(float((x.abs() / b.clamp_min(1e-300)).max()) for x, b in zip(g[:20], bars[:20]))


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_fused_mlp_every_tile_vs_float64(case):
    from mvip_nerf_b200 import _lib, ops
    name, size, mode = case
    t_start = time.time()
    dev = "cuda"
    pairs = n_pairs()
    P = size(pairs)
    T = ref.num_tiles(P)
    lib = _lib.load()
    p = orc.init_params(41)
    blob = ops.mlp_pack([torch.from_numpy(p[n]).to(dev) for n in ops.PARAM_ORDER])
    g = torch.Generator(device=dev).manual_seed(1000 + P)
    args, pts, vd = inputs(ops, P, mode, blob, g)

    # ---- forward into a NaN-filled stash ----
    s, keep = ops._points_struct(**args)
    stash = ops._aligned_bytes(lib.mvip_mlp_stash_bytes(P), dev)
    stash.fill_(0xFF)
    raw = torch.full((P, 4), float("nan"), device=dev)
    _lib.check(lib.mvip_mlp_forward(ops._ptr(blob), ctypes.byref(s), ops._ptr(raw), ops._ptr(stash), ops._stream()),
               "mvip_mlp_forward")
    del keep

    # ---- backward: poisoned workspace, NaN gradients, NaN rows after d_raw ----
    buf = torch.full((P + 64, 4), float("nan"), device=dev)
    buf[:P] = torch.randn(P, 4, device=dev, generator=g)
    d_raw = buf[:P]
    ws = ops._aligned_bytes(lib.mvip_mlp_backward_workspace_bytes(P), dev)
    flat = torch.full((N_GRADS,), float("nan"), device=dev)
    backward(lib, ops, blob, d_raw, P, stash, ws, flat)
    res = {"P": P, "tiles": T, "cta_pairs": pairs, "inputs": mode, "device": torch.cuda.get_device_name(0)}

    extra = {}
    if mode == "fine":          # accumulate=1 adds the reduced sum exactly once: g0 + G, bitwise
        g0 = torch.randn(N_GRADS, device=dev, generator=g)
        acc = g0.clone()
        backward(lib, ops, blob, d_raw, P, stash, ws, acc, accumulate=1)
        extra["accumulate_bitwise"] = bool(torch.equal(acc, g0 + flat))
    if mode == "coarse":        # one launch per phase bit (ops.kernel_timer's path) == the one-call backward, bitwise
        ph = torch.full((N_GRADS,), float("nan"), device=dev)
        backward(lib, ops, blob, d_raw, P, stash, ws, ph, phases=(1, 4, 8))
        extra["phases_bitwise"] = bool(torch.equal(ph, flat))
        backward(lib, ops, blob, d_raw, P, stash, ws, flat)         # the workspace again holds this call's dZ

    # ---- every tile, in chunks ----
    W = ref.params64(p, dev)
    fwd, chn = {}, {}
    mism, finite = 0, True
    G = A = GT = None
    for t0 in range(0, T, ref.CHUNK_TILES):
        tiles = range(t0, min(T, t0 + ref.CHUNK_TILES))
        st = ref.decode_stash(stash, P, tiles)
        finite &= st["finite"]
        mism += ref.forward_checks(st, W, ref.rows_of(pts, P, tiles), ref.rows_of(vd, P, tiles),
                                   raw[tiles.start * 128:min(P, tiles.stop * 128)], fwd)
        d = ref.rows_of(d_raw, P, tiles)
        dz = ref.decode_dz(ws, P, tiles)
        ref.chain(st, W, d, dz, chn)
        gk, ak = ref.wgrad(st, dz, d)
        gt, _ = ref.wgrad(st, ref.chain(st, W, d), d)
        G = gk if G is None else [x + y for x, y in zip(G, gk)]
        A = ak if A is None else [x + y for x, y in zip(A, ak)]
        GT = gt if GT is None else [x + y for x, y in zip(GT, gt)]
        del st, dz, d
    got = grad_views(flat)
    rel = ref.wgrad_rel(T)
    # bar-independent measures: err / (|dZ|^T |X|), per gradient tensor
    rel_abs = {n: float((x.double().reshape(y.shape) - y).abs().div(b.clamp_min(1e-300)).max())
               for n, x, y, b in zip(ref.PARAM_ORDER, got, G, A)}
    tf = {n: float((x.double().reshape(y.shape) - y).abs().max() / y.abs().max().clamp_min(1e-12))
          for n, x, y in zip(ref.PARAM_ORDER, got, GT)}
    # every tile exactly once in every weight gradient: projection of the error on each tile's contribution (second pass)
    err = [x.double().reshape(y.shape) - y for x, y in zip(got, G)]
    once = torch.cat([ref.tile_once(ref.decode_stash(stash, P, range(t0, min(T, t0 + ref.CHUNK_TILES))),
                                    ref.decode_dz(ws, P, range(t0, min(T, t0 + ref.CHUNK_TILES))), err)
                      for t0 in range(0, T, ref.CHUNK_TILES)])
    probe = {"first": 0, "last": T - 1}
    if T > 2 * pairs:
        probe["handed_out"] = 2 * pairs + (T - 2 * pairs) // 2
    contrib = {k: tile_contribution(stash, ws, d_raw, P, t, A) / rel for k, t in probe.items()}
    res.update(forward={k: v.summary() for k, v in fwd.items()}, chain={k: v.summary() for k, v in chn.items()},
               mask_mismatches=mism, stash_finite=finite, grads_finite=bool(torch.isfinite(flat).all()),
               grad_err_over_absdot=rel_abs, grad_err_over_absdot_max=max(rel_abs.values()), grad_bar=rel,
               teacher_forced_rel=max(tf.values()), tile_once_max=float(once.abs().max()),
               tile_once_argmax=int(once.abs().max(1).values.argmax()),
               tile_once_probes={k: float(once[t].abs().max()) for k, t in probe.items()},
               tile_contribution_over_bar=contrib, seconds=time.time() - t_start, **extra)
    record(name, res)

    assert finite and res["grads_finite"]
    assert mism == 0
    for stage, t in list(fwd.items()) + list(chn.items()):
        assert t.viol == 0, (stage, t.summary())
        if stage not in ("pe", "vpe", "pad", "heads"):       # the stages that are one bf16 rounding of an fp32 sum
            assert t.flips <= ref.FLIP_FRAC_MAX * t.n, (stage, t.summary())
    for n, v in rel_abs.items():
        assert v <= rel, (n, v, rel)
    for n, v in tf.items():
        assert v < GRAD_TF_RTOL, (n, v)
    assert res["tile_once_max"] <= ref.ONCE_BAR, (res["tile_once_max"], res["tile_once_argmax"])
    assert all(extra.values()), extra
