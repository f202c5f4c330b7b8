"""CPU test of the float64 stage reference (mlp_ref64): a stash and a dZ workspace ENCODED here from the layout formulas, with
the values of the CPU bf16 model, must decode exactly and pass every stage check; broken copies of them must fail."""
import numpy as np
import pytest
import torch

import mlp_ref64 as ref
from oracle import nerf_oracle as orc

P = 300                  # three tiles, the last one ragged (44 valid rows)
T = ref.num_tiles(P)


# ---- encoder, written from the formulas of csrc/common.cuh (chunk_off16) and csrc/mlp_common.cuh -------------------------------
def chunk_off(r, k):
    return (r >> 3) * 1024 + (r & 7) * 128 + (((k >> 3) ^ (r & 7)) << 4) + (k & 7) * 2


def mask_bit_of_column(j):
    return 16 * (j & 1) + 8 * (j >> 4) + ((j & 15) >> 1)


def mask_word_index(layer, r, h, ch):
    return layer * 1024 + ch * 512 + r * 4 + h * 2


def bf16_bits(x):
    a = np.ascontiguousarray(x, dtype=np.float32).view(np.uint32)
    assert np.array_equal(a & 0xFFFF, np.zeros_like(a)), "value is not bf16-representable"
    return (a >> 16).astype(np.uint16)


def encode_image(block):
    """[128, 64] bf16-exact values -> the 16 KB chunk image"""
    out = np.zeros(8192, np.uint16)
    bits = bf16_bits(block)
    for r in range(128):
        for k in range(64):
            out[chunk_off(r, k) // 2] = bits[r, k]
    return out.view(np.uint8)


def encode_tile(chunks, n_bytes):
    """list of [128, 64] blocks -> one tile's bytes (chunk images back to back, zero tail)"""
    out = np.zeros(n_bytes, np.uint8)
    for c, blk in enumerate(chunks):
        out[c * ref.ACT_CHUNK:(c + 1) * ref.ACT_CHUNK] = encode_image(blk)
    return out


def split64(x):
    x = np.pad(x, ((0, 0), (0, (-x.shape[1]) % 64)))
    return [x[:, 64 * j:64 * j + 64] for j in range(x.shape[1] // 64)]


def encode_masks(layers):
    """9 bool [128, 256 | 128] masks -> the 9 x 4 KB mask block"""
    words = np.zeros(9 * 1024, np.uint32)
    for layer, m in enumerate(layers):
        for c in range(m.shape[1]):
            h, ch, i, j = c >> 7, (c >> 6) & 1, (c >> 5) & 1, c & 31
            for r in np.nonzero(m[:, c])[0]:
                words[mask_word_index(layer, r, h, ch) + i] |= np.uint32(1) << np.uint32(mask_bit_of_column(j))
    return words.view(np.uint8)


def model():
    rng = np.random.RandomState(31)
    p = orc.init_params(17)
    pts = np.zeros((T * 128, 3), np.float32)              # rows past P: the zero point the forward encodes there
    vd = np.zeros((T * 128, 3), np.float32)
    d_raw = np.zeros((T * 128, 4), np.float32)            # ... and a zero upstream gradient
    pts[:P] = (rng.rand(P, 3) * 2 - 1) * 3
    vd[:P] = rng.randn(P, 3)
    vd[:P] /= np.linalg.norm(vd[:P], axis=-1, keepdims=True)
    d_raw[:P] = rng.randn(P, 4)
    out, g, k = orc.nerf_forward_backward_bf16sim(p, pts, vd, d_raw, keep=True)
    return p, pts, vd, d_raw, out, g, k


def encode(k):
    stash, dz = [], []
    for t in range(T):
        s = slice(128 * t, 128 * t + 128)
        chunks = split64(k["pe"][s]) + sum([split64(h[s]) for h in k["h"]], []) + split64(k["feat"][s]) + \
            split64(k["vpe"][s]) + split64(k["hidden"][s])
        tile = encode_tile(chunks, ref.STASH_TILE_BYTES)
        tile[ref.STASH_MASK_OFF:] = encode_masks([h[s] > 0 for h in k["h"]] + [k["hidden"][s] > 0])
        stash.append(tile)
        chunks = split64(k["d_hidden_pre"][s]) + split64(k["d_feat"][s]) + sum([split64(k["dz"][7 - t_][s]) for t_ in range(8)], [])
        dz.append(encode_tile(chunks, ref.DZ_TILE_BYTES))
    return torch.from_numpy(np.concatenate(stash)), torch.from_numpy(np.concatenate(dz))


@pytest.fixture(scope="module")
def case():
    p, pts, vd, d_raw, out, g, k = model()
    stash, dz = encode(k)
    return dict(p=p, pts=pts, vd=vd, d_raw=d_raw, out=out, g=g, k=k, stash=stash, dz=dz, W=ref.params64(p, "cpu"))


def run_checks(c, stash, dz, skip_tile=None):
    """-> (forward tallies, mask mismatches, chain tallies, per-tensor gradient excess over the wgrad_rel bar, max rel diff,
    [tiles, 10] projections of the gradient error on each tile's contribution)"""
    fwd, chn, tot, bars = {}, {}, None, None
    mism = 0
    for t in range(T):
        tiles = range(t, t + 1)
        st = ref.decode_stash(stash, P, tiles)
        d = ref.rows_of(torch.from_numpy(c["d_raw"][:P]), P, tiles)
        raw = ref.rows_of(torch.from_numpy(c["out"][:P]), P, tiles)
        mism += ref.forward_checks(st, c["W"], torch.from_numpy(c["pts"][128 * t:128 * t + 128]).double(),
                                   torch.from_numpy(c["vd"][128 * t:128 * t + 128]).double(), raw, fwd)
        dzt = ref.decode_dz(dz, P, tiles)
        ref.chain(st, c["W"], d, dzt, chn)
        if t == skip_tile:
            continue
        g, a = ref.wgrad(st, dzt, d)
        tot = g if tot is None else [x + y for x, y in zip(tot, g)]
        bars = a if bars is None else [x + y for x, y in zip(bars, a)]
    want = [torch.from_numpy(np.asarray(c["g"][n], dtype=np.float64)) for n in ref.PARAM_ORDER]
    want = [w.reshape(x.shape) for w, x in zip(want, tot)]
    rel = max(float((x - w).abs().max() / w.abs().max()) for x, w in zip(tot, want))
    # a model with a tile left out: the bf16 model's gradients play the kernel's part, tot the float64 sum
    err = [w - x for x, w in zip(tot, want)]
    once = torch.cat([ref.tile_once(ref.decode_stash(stash, P, range(t, t + 1)), ref.decode_dz(dz, P, range(t, t + 1)), err)
                      for t in range(T)])
    return fwd, mism, chn, ref.grad_excess(tot, want, bars, ref.wgrad_rel(T)), rel, once


def test_decode_gives_back_what_was_encoded(case):
    k = case["k"]
    st = ref.decode_stash(case["stash"], P, range(0, T))
    assert st["finite"]
    assert torch.equal(st["pe"][:, :63], torch.from_numpy(k["pe"])) and torch.equal(st["vpe"][:, :27], torch.from_numpy(k["vpe"]))
    assert float(st["pe"][:, 63:].abs().max()) == 0 and float(st["vpe"][:, 27:].abs().max()) == 0
    for l in range(8):
        assert torch.equal(st["h"][l], torch.from_numpy(k["h"][l])), l
        assert torch.equal(st["mask"][l], torch.from_numpy(k["h"][l] > 0)), l
    assert torch.equal(st["feat"], torch.from_numpy(k["feat"])) and torch.equal(st["hidden"], torch.from_numpy(k["hidden"]))
    assert torch.equal(st["mask"][8], torch.from_numpy(k["hidden"] > 0))
    assert int(st["valid"].sum()) == P and bool(st["valid"][:P].all())
    dz = ref.decode_dz(case["dz"], P, range(0, T))
    assert torch.equal(dz["hidden"], torch.from_numpy(k["d_hidden_pre"])) and torch.equal(dz["feat"], torch.from_numpy(k["d_feat"]))
    for l in range(8):
        assert torch.equal(dz["z"][l], torch.from_numpy(k["dz"][l])), l
    # a sub-range decodes to the same rows
    st1 = ref.decode_stash(case["stash"], P, range(1, 3))
    assert torch.equal(st1["h"][3], st["h"][3][128:]) and torch.equal(st1["mask"][8], st["mask"][8][128:])


def test_stage_checks_pass_on_the_bf16_model(case):
    fwd, mism, chn, excess, rel, once = run_checks(case, case["stash"], case["dz"])
    assert mism == 0
    assert set(fwd) == {"pe", "vpe", "pad", "heads", "feature", "hidden"} | {"L%d" % l for l in range(8)}
    assert set(chn) == {"d_hidden_pre", "d_feature"} | {"dZ%d" % l for l in range(8)}
    for name, t in list(fwd.items()) + list(chn.items()):
        assert t.viol == 0, (name, t.summary())
        if name not in ("pe", "vpe", "heads"):
            assert t.flips == 0, (name, t.summary())     # the same float64 sums, rounded once: identical bf16
    assert rel < 1e-12, rel
    assert max(excess) < 1e-3, excess
    assert float(once.abs().max()) < 1e-9, once


def test_teacher_forced_grads_equal_the_bf16_model(case):
    g = ref.teacher_forced_grads(case["p"], case["stash"], P, torch.from_numpy(case["d_raw"][:P]))
    for n in ref.PARAM_ORDER:
        want = np.asarray(case["g"][n], dtype=np.float64)
        assert float(np.abs(g[n].numpy().reshape(want.shape) - want).max()) <= 1e-12 * float(np.abs(want).max()), n


# ---- mutations: each must make a check fail ---------------------------------------------------------------------------------
def _row_bytes(tile, chunk, r):
    base = tile * ref.STASH_TILE_BYTES + chunk * ref.ACT_CHUNK
    return [base + chunk_off(r, k) + b for k in range(64) for b in range(2)]


def test_swapped_rows_of_h3_fail_the_forward_check(case):
    stash = case["stash"].clone()
    for chunk in range(1 + 4 * 2, 5 + 4 * 2):              # h3 = output of pts_linears.2: chunks 9..12
        a, b = _row_bytes(1, chunk, 5), _row_bytes(1, chunk, 70)
        stash[a], stash[b] = case["stash"][b], case["stash"][a]
    fwd = run_checks(case, stash, case["dz"])[0]
    assert fwd["L2"].viol > 0 and fwd["L3"].viol > 0


def test_flipped_mask_bit_fails_the_checks(case):
    k = case["k"]
    l, r, c = 3, 17, None
    for c in range(256):                                   # a live unit whose dZ is non-zero
        if k["h"][l][128 + r, c] > 0 and k["dz"][l][128 + r, c] != 0:
            break
    h, ch, i, j = c >> 7, (c >> 6) & 1, (c >> 5) & 1, c & 31
    off = ref.STASH_TILE_BYTES + ref.STASH_MASK_OFF + 4 * (mask_word_index(l, r, h, ch) + i) + mask_bit_of_column(j) // 8
    stash = case["stash"].clone()
    stash[off] ^= 1 << (mask_bit_of_column(j) % 8)
    fwd, mism, chn = run_checks(case, stash, case["dz"])[:3]
    assert mism == 1
    assert chn["dZ%d" % l].viol > 0


def test_dropped_tile_fails_the_gradient_check(case):
    _, _, _, excess, rel, once = run_checks(case, case["stash"], case["dz"], skip_tile=1)
    assert rel > 1e-3
    # every weight / bias gradient the fused backward produces would be outside its bar
    assert min(excess[:20]) > 10, excess
    # ... and so would the every-tile-once projection: the "kernel" (the bf16 model) counts tile 1 once more than the sum
    # does, in all ten weight gradients: +1 exactly (the other tiles' contributions are not orthogonal to it, so they see it too)
    assert torch.allclose(once[1], torch.ones(10, dtype=torch.float64), atol=1e-9), once[1]
    assert float(once.abs().max()) > ref.ONCE_BAR
