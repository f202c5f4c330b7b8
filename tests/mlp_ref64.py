"""Float64 reference of the fused NeRF MLP, stage by stage, from the bytes the kernels keep (torch; runs on cuda or cpu).

The forward stash holds the exact bf16 operands every MMA of the forward consumed, and the backward workspace holds the exact
bf16 dZ images the dgrad chain published.  Each stage of every tile can therefore be recomputed in float64 from its own inputs:
what is left between the kernel and this reference is fp32 accumulation and one bf16 rounding, so the bars are one bf16 ulp
(plus a floor for values within fp32-accumulation error of zero) rather than an end-to-end fraction of the tensor's max.

Layouts (cited, not restated):
  * chunk image: 128 rows x 64 bf16, 128-byte swizzle = chunk_off16 (csrc/common.cuh), DESIGN.md section 3;
  * forward stash per tile: 40 chunk images, then 9 x 4 KB of ReLU mask words: kStash* and mask_word_index /
    mask_bit_of_column in csrc/mlp_common.cuh;
  * dZ images per tile at workspace offset 0 (carve() in csrc/mlp_backward.cu), 38 chunk images: 0-1 d hidden_pre,
    2-5 d feature, 6 + 4 t + j = dZ of layer 7 - t (kDz* in csrc/mlp_common.cuh).
Operand roundings are those of oracle.nerf_forward_backward_bf16sim: MMA weights bf16; biases, the alpha / rgb head weights and
d_raw fp32; the forward heads read the fp32 activations, the backward heads the bf16 stash rows.
"""
import torch

TILE = 128
ACT_CHUNK = 128 * 128                       # bytes of one chunk image
STASH_MASK_OFF = 40 * ACT_CHUNK
STASH_TILE_BYTES = STASH_MASK_OFF + 9 * 128 * 32
DZ_TILE_BYTES = 38 * ACT_CHUNK
CHUNK_TILES = 256                           # tiles per decode: 32,768 points, ~1.3 GB of float64 at a time

PARAM_ORDER = (["pts_linears.%d.%s" % (i, k) for i in range(8) for k in ("weight", "bias")] +
               ["views_linears.0.weight", "views_linears.0.bias", "feature_linear.weight", "feature_linear.bias",
                "alpha_linear.weight", "alpha_linear.bias", "rgb_linear.weight", "rgb_linear.bias"])

# ---- bars (B200 measurements in profiles/r03_mlp_fullsize.json, DESIGN.md section 2) ----------------------------------------
# fp32 accumulation error of one MMA output, relative to sum |x||w| (+|b|): the floor added to the one-ulp bar.  A K <= 320
# fp32 sum is exact to ~K * 2^-24 of that sum in the worst case; 2^-17 leaves the one-ulp bar in force for every value larger
# than ~2^-9 of its |x||w| sum.
ACC_FLOOR = 2.0 ** -17
# fraction of elements per stage whose bf16 differs by one ulp from the float64 rounding (fp32 sums that land on the other
# side of a rounding boundary).  Measured on a B200 at 21 sizes from 1 to 2^21 + 3 points: at most 1.8e-4 (hidden, dZ4).
FLIP_FRAC_MAX = 4e-4
# weight / bias gradients: |kernel - float64| <= wgrad_rel(tiles) * (|dZ|^T |X|) elementwise.  What is left is the fp32 order of
# the sums: within a tile (the MMA's K = 128 points) and over the tiles a CTA pair accumulates in tensor memory and the reduce
# adds, which grows like sqrt(tiles).  Measured on a B200: 2.2e-7 at one tile, 1.1e-6 at 2,048 tiles, 4.6e-6 at 16,385; the bar
# is the fit a + b sqrt(tiles) of those maxima, doubled (the measured maxima sit at 0.09 - 0.43 of it).
WGRAD_A, WGRAD_B = 5e-7, 8e-8
# every tile exactly once in every weight gradient of the fused backward: the projection of the kernel's error on one tile's
# float64 contribution, <err, C_t> / <C_t, C_t>, is -1 for a dropped tile and +1 for a double-counted one.  What fp32 order
# leaves is noise over |C_t|: measured on a B200 at most 0.045 for a full tile (1,572,875 points), 0.161 for the 3-point last
# tile of 2^21 + 3 points (1/40 of a full tile's contribution); the bar is about twice that.
ONCE_BAR = 0.35
# forward heads: the kernel's heads read the fp32 activations, the stash holds their bf16 rounding (relative 2^-8 at most)
HEAD_REL, HEAD_ABS = 2.0 ** -8, 1e-5
PE_ATOL, VPE_ATOL = 8e-3, 2e-2               # the bars of test_gpu_mlp.test_stash_matches_bf16_model


def num_tiles(P):
    return (P + TILE - 1) // TILE


def wgrad_rel(tiles):
    return WGRAD_A + WGRAD_B * tiles ** 0.5


def bf16(x):
    """float64 -> fp32 -> bf16 (round to nearest even) -> float64, as oracle.bf16_round"""
    return x.float().bfloat16().double()


def bf16_ulp(a):
    """spacing of bf16 numbers at |a| (a >= 0, bf16-representable magnitudes); 0 at a = 0"""
    _, e = torch.frexp(a)
    return torch.where(a > 0, torch.ldexp(torch.ones_like(a), e - 8), torch.zeros_like(a))


def params64(p, device):
    """{name: fp32 array / tensor} -> float64 tensors: MMA weights rounded to bf16, biases and the head weights kept fp32"""
    out = {}
    for k, v in p.items():
        t = torch.as_tensor(v).to(device=device, dtype=torch.float32)
        if k.endswith("weight") and not k.startswith(("alpha", "rgb")):
            t = t.bfloat16()
        out[k] = t.double()
    return out


# ---- decoding ------------------------------------------------------------------------------------------------------------------
_IDX = {}


def _image_index(device):
    """(row, col) -> u16 index inside a chunk image: chunk_off16 of common.cuh, (r>>3)*1024 + (r&7)*128 + ((k>>3 ^ r&7)<<4) + (k&7)*2"""
    key = str(device)
    if key not in _IDX:
        r = torch.arange(128).view(128, 1)
        k = torch.arange(64).view(1, 64)
        off = (r >> 3) * 1024 + (r & 7) * 128 + (((k >> 3) ^ (r & 7)) << 4) + (k & 7) * 2
        c = torch.arange(256).view(1, 256)      # mask: column c = 128 h + 64 ch + 32 i + j
        h, ch, i, j = c >> 7, (c >> 6) & 1, (c >> 5) & 1, c & 31
        word = ch * 512 + r * 4 + h * 2 + i                                   # mask_word_index(0, r, h, ch) + i
        bit = 16 * (j & 1) + 8 * (j >> 4) + ((j & 15) >> 1)                   # mask_bit_of_column(j)
        _IDX[key] = ((off // 2).reshape(-1).to(device), word.reshape(-1).to(device), bit.expand(128, 256).reshape(-1).to(device))
    return _IDX[key]


def _images(buf_u8, tile_bytes, n_chunks, tiles):
    """-> float64 [n_tiles, n_chunks, 128, 64]: the chunk images of the tile range, unswizzled"""
    t0, t1 = tiles.start, tiles.stop
    raw = buf_u8[t0 * tile_bytes:t1 * tile_bytes].view(t1 - t0, tile_bytes)[:, :n_chunks * ACT_CHUNK]
    u16 = raw.view(torch.int16).reshape(t1 - t0, n_chunks, ACT_CHUNK // 2)
    idx = _image_index(buf_u8.device)[0]
    return (u16[:, :, idx].to(torch.int32) << 16).view(torch.float32).double().view(t1 - t0, n_chunks, 128, 64)


def _cols(img, a, b):
    """chunk images a..b-1 side by side -> [n_tiles * 128, 64 (b - a)]"""
    n = img.shape[0]
    return img[:, a:b].permute(0, 2, 1, 3).reshape(n * 128, 64 * (b - a))


def _check_range(P, tiles):
    assert tiles.step == 1 and 0 <= tiles.start < tiles.stop <= num_tiles(P), (P, tiles)


def decode_stash(stash_u8, P, tiles):
    """Forward stash of the tile range -> float64 [rows, feat] tensors and bool ReLU masks; rows = 128 per tile, the rows past
    P of the last tile included.  pe / vpe: the whole 64-column chunk (pad columns too); h[l]: output of pts_linears.l;
    mask[l] (l < 8): ReLU mask of h[l], mask[8]: of hidden; valid: row < P."""
    _check_range(P, tiles)
    img = _images(stash_u8, STASH_TILE_BYTES, 40, tiles)
    n = tiles.stop - tiles.start
    st = {"pe": _cols(img, 0, 1), "h": [_cols(img, 1 + 4 * l, 5 + 4 * l) for l in range(8)], "feat": _cols(img, 33, 37),
          "vpe": _cols(img, 37, 38), "hidden": _cols(img, 38, 40)}
    _, word, bit = _image_index(stash_u8.device)
    t0, t1 = tiles.start, tiles.stop
    words = stash_u8[t0 * STASH_TILE_BYTES:t1 * STASH_TILE_BYTES].view(n, STASH_TILE_BYTES)[:, STASH_MASK_OFF:]
    words = words.view(torch.int32).reshape(n, 9, 1024)
    bits = ((words[:, :, word] >> bit) & 1).bool().view(n, 9, 128, 256).permute(1, 0, 2, 3).reshape(9, n * 128, 256)
    st["mask"] = [bits[l] for l in range(8)] + [bits[8][:, :128]]
    st["valid"] = torch.arange(t0 * TILE, t1 * TILE, device=stash_u8.device) < P
    st["finite"] = bool(torch.isfinite(img).all())
    return st


def decode_dz(ws_u8, P, tiles):
    """dZ images the dgrad chain published, for the tile range -> float64 [rows, feat]: hidden = d hidden_pre,
    feat = d feature, z[l] = dZ of pts_linears.l"""
    _check_range(P, tiles)
    img = _images(ws_u8, DZ_TILE_BYTES, 38, tiles)
    return {"hidden": _cols(img, 0, 2), "feat": _cols(img, 2, 6), "z": [_cols(img, 6 + 4 * (7 - l), 10 + 4 * (7 - l)) for l in range(8)]}


def rows_of(x, P, tiles):
    """rows [128 t0, 128 t1) of a [P, c] tensor as float64, zeros past P (what the kernels see for the padding rows)"""
    r0, r1 = tiles.start * TILE, tiles.stop * TILE
    out = torch.zeros((r1 - r0, x.shape[1]), dtype=torch.float64, device=x.device)
    out[:max(0, min(P, r1) - r0)] = x[r0:min(P, r1)].double()
    return out


# ---- stage checks --------------------------------------------------------------------------------------------------------------
class Tally:
    """violations of a bar, one-ulp flips and the worst err / bar of one stage over many tiles"""

    def __init__(self):
        self.n = self.viol = self.flips = 0
        self.worst = 0.0

    def add(self, got, ref, tol):
        err = (got - ref).abs()
        self.n += got.numel()
        self.viol += int((~(err <= tol)).sum())                  # NaN counts as a violation
        self.flips += int((got != ref).sum())
        ratio = torch.where(err == 0, torch.zeros_like(err), err / tol)
        self.worst = max(self.worst, float(torch.nan_to_num(ratio, nan=float("inf")).max()))

    def summary(self):
        return {"n": self.n, "violations": self.viol, "flip_frac": self.flips / max(self.n, 1), "worst_err_over_bar": self.worst}


def _rounding_stage(tally, got, pre, absacc):
    """got = bf16 of an fp32 sum whose float64 value is pre: one bf16 ulp + the fp32-accumulation floor"""
    ref = bf16(pre)
    tol = bf16_ulp(torch.maximum(got.abs(), ref.abs())) + ACC_FLOOR * absacc
    tally.add(got, ref, tol)


def embed64(x, L):
    """positional encoding in float64 of fp32 inputs: [x, sin(2^k x), cos(2^k x), ...] (oracle.embed's column order)"""
    outs = [x]
    for k in range(L):
        outs += [torch.sin(x * 2.0 ** k), torch.cos(x * 2.0 ** k)]
    return torch.cat(outs, 1)


def trunk_input(st, l):
    """operand of pts_linears.l as the forward fed it: PE, [PE | h4] for the skip layer, else the previous output"""
    if l == 0:
        return st["pe"][:, :63]
    if l == 5:
        return torch.cat([st["pe"][:, :63], st["h"][4]], 1)
    return st["h"][l - 1]


def views_input(st):
    return torch.cat([st["feat"], st["vpe"][:, :27]], 1)


def _linear(x, w, b):
    return x @ w.T + b, x.abs() @ w.abs().T + b.abs()


def forward_checks(st, W, pts, vd, raw, tallies):
    """Every stage of the forward for the decoded rows.  pts / vd: float64 of the fp32 inputs (zeros past P); raw: the kernel's
    [rows, 4] output (only rows < P are compared).  Fills tallies[stage] and returns the number of mask mismatches."""
    t = tallies
    _tally(t, "pe").add(st["pe"][:, :63], bf16(embed64(pts, 10)), torch.full_like(st["pe"][:, :63], PE_ATOL))
    _tally(t, "vpe").add(st["vpe"][:, :27], bf16(embed64(vd, 4)), torch.full_like(st["vpe"][:, :27], VPE_ATOL))
    _tally(t, "pad").add(torch.cat([st["pe"][:, 63:], st["vpe"][:, 27:]], 1), 0.0, 0.0)
    for l in range(8):
        pre, absacc = _linear(trunk_input(st, l), W["pts_linears.%d.weight" % l], W["pts_linears.%d.bias" % l])
        _rounding_stage(_tally(t, "L%d" % l), st["h"][l], pre.clamp_min(0), absacc)
    pre, absacc = _linear(st["h"][7], W["feature_linear.weight"], W["feature_linear.bias"])
    _rounding_stage(_tally(t, "feature"), st["feat"], pre, absacc)
    pre, absacc = _linear(views_input(st), W["views_linears.0.weight"], W["views_linears.0.bias"])
    _rounding_stage(_tally(t, "hidden"), st["hidden"], pre.clamp_min(0), absacc)
    mism = sum(int((st["mask"][l] != (st["h"][l] > 0)).sum()) for l in range(8))
    mism += int((st["mask"][8] != (st["hidden"] > 0)).sum())
    rgb, rgb_abs = _linear(st["hidden"], W["rgb_linear.weight"], W["rgb_linear.bias"])
    alpha, alpha_abs = _linear(st["h"][7], W["alpha_linear.weight"], W["alpha_linear.bias"])
    v = st["valid"][:raw.shape[0]]
    want = torch.cat([rgb, alpha], 1)[:raw.shape[0]][v]
    bar = HEAD_REL * torch.cat([rgb_abs, alpha_abs], 1)[:raw.shape[0]][v] + HEAD_ABS
    _tally(t, "heads").add(raw[v].double(), want, bar)
    return mism


def _tally(t, name):
    if name not in t:
        t[name] = Tally()
    return t[name]


def chain(st, W, d_raw, dz=None, tallies=None):
    """The dgrad chain in float64 with the kernels' roundings.  dz is None: the teacher-forced model, every step from its own
    bf16 output; returns its dZ images (decode_dz's layout).  dz given (the kernel's images): every step is recomputed from the
    kernel's OWN previous dZ and compared with the kernel's output into tallies."""
    m = [x.double() for x in st["mask"]]
    d_rgb, d_alpha = d_raw[:, :3], d_raw[:, 3:4]
    kern = dz if dz is not None else {"hidden": None, "feat": None, "z": [None] * 8}

    def step(name, pre, absacc, mask, got):
        """-> this step's dZ as the next step consumes it: the model's bf16 rounding, or the kernel's own image"""
        if mask is not None:
            pre, absacc = pre * mask, absacc * mask
        if dz is None:
            return bf16(pre)
        _rounding_stage(_tally(tallies, name), got, pre, absacc)
        return got

    out = {"z": [None] * 8}
    wr = W["rgb_linear.weight"]                                        # fp32: the input stage runs on CUDA cores
    dh = out["hidden"] = step("d_hidden_pre", d_rgb @ wr, d_rgb.abs() @ wr.abs(), m[8], kern["hidden"])
    wv = W["views_linears.0.weight"][:, :256]
    df = out["feat"] = step("d_feature", dh @ wv, dh.abs() @ wv.abs(), None, kern["feat"])
    wf, wa = W["feature_linear.weight"], W["alpha_linear.weight"]
    d = step("dZ7", df @ wf + d_alpha @ wa, df.abs() @ wf.abs() + d_alpha.abs() @ wa.abs(), m[7], kern["z"][7])
    out["z"][7] = d
    for l in reversed(range(7)):
        w = W["pts_linears.%d.weight" % (l + 1)]
        if l == 4:
            w = w[:, 63:]                                              # the h4 part of [PE | h4]
        d = out["z"][l] = step("dZ%d" % l, d @ w, d.abs() @ w.abs(), m[l], kern["z"][l])
    return out


def wgrad(st, dz, d_raw):
    """-> (grads, bars): float64 gradients of the rows in PARAM_ORDER from the stash and dZ images, and the matching
    |dZ|^T |X| (column sums of |dZ| for biases), the scale of fp32 accumulation-order error"""
    g, a = {}, {}

    def acc(name, d, x):
        g[name + ".weight"], a[name + ".weight"] = d.T @ x, d.abs().T @ x.abs()
        g[name + ".bias"], a[name + ".bias"] = d.sum(0), d.abs().sum(0)

    for l in range(8):
        acc("pts_linears.%d" % l, dz["z"][l], trunk_input(st, l))
    acc("views_linears.0", dz["hidden"], views_input(st))
    acc("feature_linear", dz["feat"], st["h"][7])
    acc("alpha_linear", d_raw[:, 3:4], st["h"][7])
    acc("rgb_linear", d_raw[:, :3], st["hidden"])
    return [g[n] for n in PARAM_ORDER], [a[n] for n in PARAM_ORDER]


def teacher_forced_grads(p, stash_u8, P, d_raw):
    """float64 backward of the whole batch from the decoded stash alone (the chain recomputed, not read back):
    {name: tensor} in PARAM_ORDER"""
    dev = stash_u8.device
    W = params64(p, dev)
    d_raw = torch.as_tensor(d_raw).to(dev).reshape(-1, 4)
    tot = None
    for t0 in range(0, num_tiles(P), CHUNK_TILES):
        tiles = range(t0, min(num_tiles(P), t0 + CHUNK_TILES))
        st = decode_stash(stash_u8, P, tiles)
        d = rows_of(d_raw, P, tiles)
        g, _ = wgrad(st, chain(st, W, d), d)
        tot = g if tot is None else [x + y for x, y in zip(tot, g)]
    return dict(zip(PARAM_ORDER, tot))


def grad_excess(got, want, bars, rel):
    """per tensor: max |got - want| / (rel * bar) (> 1: outside the bar; NaN -> inf)"""
    out = []
    for x, y, b in zip(got, want, bars):
        err = (x.double().reshape(y.shape) - y).abs()
        r = torch.where(err == 0, torch.zeros_like(err), err / (rel * b))
        out.append(float(torch.nan_to_num(r, nan=float("inf")).max()))
    return out


FUSED_WEIGHTS = [PARAM_ORDER.index(n) for n in PARAM_ORDER[:20] if n.endswith("weight")]   # pts_linears 0..7, views, feature


def tile_once(st, dz, err):
    """-> [n_tiles, 10]: for each tile of the range and each weight gradient of the fused backward, the projection
    <err, C_t> / <C_t, C_t> of the kernel's error err (kernel - float64 sum, PARAM_ORDER) on the tile's float64
    contribution C_t = dZ_t^T X_t.  ~0 when every tile is counted once; -1 when tile t is missing, +1 when it is counted twice
    (tiles' contributions are not orthogonal: such an error shows on the neighbouring tiles' projections as well)."""
    n = st["h"][0].shape[0] // TILE
    ops = [(dz["z"][l], trunk_input(st, l)) for l in range(8)] + [(dz["hidden"], views_input(st)), (dz["feat"], st["h"][7])]
    out = []
    for (d, x), i in zip(ops, FUSED_WEIGHTS):
        e = err[i].reshape(d.shape[1], x.shape[1])
        num = (d * (x @ e.T)).sum(1).view(n, TILE).sum(1)                           # sum over rows of d_r . (E x_r)
        c = torch.bmm(d.view(n, TILE, -1).transpose(1, 2), x.view(n, TILE, -1))      # C_t
        den = c.pow(2).sum((1, 2))
        out.append(torch.where(den > 0, num / den.clamp_min(1e-300), torch.zeros_like(num)))
    return torch.stack(out, 1)
