"""The tensor-core weight gradient walks only live (row chunk, offset group) items, balances its row splits by live items,
and the BatchNorm backward pass sums the bias gradient of the convolution in front of it.

Weight gradient: with the rulebook's tile masks the kernel skips every group of 128/Cin kernel offsets (a "pass") that has
no neighbour in a row chunk's 128-row tile, skips chunks with no live pass whole, and gives each CTA a row range holding
an equal share of its offset group's live items, computed on the device.  toda_spconv_wgrad_row_splits reports those
ranges, so the tests below place live items relative to the ranges the library really uses.  Results must match a
float64 reference and be bit-identical from run to run.  Synthetic tables put the live items where the kernel's
hand-offs are most fragile: splits with no live item, a pass live only in a split's last chunk, one live pass per chunk
(the dy-buffer ring then drains), for 128-row chunks (Cout <= 64) and 64-row chunks (Cout = 128).

Bias gradient: sum_rows dy, accumulated in fixed-order fp64 by the pass that writes dy, against a float64 sum of the fp32
dy that pass wrote; the fused layer call and the stepwise calls give the same bits.
"""
import ctypes

import numpy as np
import pytest
import torch

from tests import test_gpu_layers as TL
from tests.test_gpu_layers import full  # noqa: F401  (module fixture: every conv geometry of VoxelResBackBone8x)

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _ops():
    from toda_b200 import ops
    return ops


def _row_splits(masks, n_out, kvol, cin, cout):
    """[groups][splits + 1] row boundaries of the wgrad launch, as the library computes them from the masks."""
    from toda_b200 import _C
    ops = _ops()
    L = _C.lib()
    groups, splits = ctypes.c_int(), ctypes.c_int()
    _C.check(L.toda_spconv_wgrad_row_splits(None, n_out, kvol, cin, cout, ctypes.byref(groups), ctypes.byref(splits), None,
                                            None), "toda_spconv_wgrad_row_splits")
    rb = torch.empty((groups.value * splits.value,), dtype=torch.int32, device=DEV)
    _C.check(L.toda_spconv_wgrad_row_splits(masks.data_ptr() if masks is not None else None, n_out, kvol, cin, cout,
                                            ctypes.byref(groups), ctypes.byref(splits), rb.data_ptr(), ops._stream()),
             "toda_spconv_wgrad_row_splits")
    b = rb.view(groups.value, splits.value).cpu().numpy().astype(np.int64)
    return np.concatenate([b, np.full((groups.value, 1), n_out, np.int64)], 1)


def _chunk_rows(cout):
    return 128 if cout <= 64 else 64


def _wgrad(x, xb, nbr, n_out, kvol, dy, dyb, cout, masks):
    """toda_spconv_wgrad in bf16 -> dw in the parameter layout (cout, kvol, cin)."""
    from toda_b200 import _C
    ops = _ops()
    L = _C.lib()
    n_in, cin = x.shape
    dw = torch.empty((cout, kvol, cin), dtype=torch.float32, device=DEV)
    ws = torch.empty((L.toda_spconv_wgrad_workspace_bytes(n_in, n_out, kvol, cin, cout, ops.CONV_BF16),), dtype=torch.uint8,
                     device=DEV)
    p = lambda t: t.data_ptr() if t is not None else None  # noqa: E731
    _C.check(L.toda_spconv_wgrad(p(x), p(xb), n_in, cin, p(nbr), n_out, kvol, p(masks), p(dy), p(dyb), cout, p(dw), p(ws),
                                 ws.numel(), ops.CONV_BF16, ops._stream()), "toda_spconv_wgrad")
    torch.cuda.synchronize()
    return dw


def _ref_wgrad(x, nbr, dy):
    """float64 dw[co, k, ci] = sum_o x[nbr[k, o], ci] * dy[o, co]."""
    kvol = nbr.shape[0]
    xd, dyd = x.double(), dy.double()
    out = torch.zeros((dy.shape[1], kvol, x.shape[1]), dtype=torch.float64, device=DEV)
    for k in range(kvol):
        o = torch.nonzero(nbr[k] >= 0).flatten()
        if o.numel():
            out[:, k, :] = dyd[o].t() @ xd[nbr[k, o].long()]
    return out


def _operands(n_in, n_out, cin, cout, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    x = TL.bf16_round(torch.randn((n_in, cin), device=DEV, generator=g))
    dy = TL.bf16_round(torch.randn((n_out, cout), device=DEV, generator=g))
    return x, x.to(torch.bfloat16), dy, dy.to(torch.bfloat16)


def _table(n_in, n_out, kvol, live, seed, density=0.3):
    """int32 [kvol][n_out] table: a neighbour at random rows wherever live(k, row) holds, -1 elsewhere."""
    rng = np.random.default_rng(seed)
    ks, rows = np.meshgrid(np.arange(kvol), np.arange(n_out), indexing="ij")
    keep = live(ks, rows) & (rng.random((kvol, n_out)) < density)
    nbr = np.where(keep, rng.integers(0, n_in, (kvol, n_out)), -1).astype(np.int32)
    return torch.from_numpy(nbr).to(DEV)


def _check_live(nbr, n_in, cin, cout, seed, what):
    """Two runs bit-identical; masks and NULL masks both against the float64 reference.  -> the masks."""
    ops = _ops()
    kvol, n_out = nbr.shape
    x, xb, dy, dyb = _operands(n_in, n_out, cin, cout, seed)
    masks = ops.table_tile_masks(nbr)
    a = _wgrad(x, xb, nbr, n_out, kvol, dy, dyb, cout, masks)
    b = _wgrad(x, xb, nbr, n_out, kvol, dy, dyb, cout, masks)
    full_walk = _wgrad(x, xb, nbr, n_out, kvol, dy, dyb, cout, None)
    assert torch.equal(a, b), f"{what}: two runs differ"
    ref = _ref_wgrad(x, nbr, dy)
    TL.check(a, ref, what=what)
    TL.check(full_walk, ref, what=what + " (NULL masks)")
    return masks


def _live_chunks(masks, n_out, rows, k0, opp):
    """bool per row chunk: the pass of offsets [k0, k0 + opp) has a neighbour in the chunk's 128-row tile."""
    m = masks.cpu().numpy().astype(np.int64) & 0xFFFFFFFF
    word = m[(np.arange((n_out + rows - 1) // rows) * rows) >> 7]
    return ((word >> k0) & ((1 << opp) - 1)) != 0


@pytest.mark.parametrize("cin,cout", [(16, 32), (32, 64), (64, 128), (128, 128)])
def test_splits_without_live_items(cin, cout):
    """Neighbours in the first three tiles only: fewer live items than splits, so most CTAs walk no item and must leave a
    zero partial."""
    n_in, n_out, kvol = 5000, 40000, 27
    nbr = _table(n_in, n_out, kvol, lambda k, r: (r < 384) & (k == 0), seed=1, density=0.5)
    masks = _check_live(nbr, n_in, cin, cout, 11, f"three live tiles {cin}->{cout}")
    b = _row_splits(masks, n_out, kvol, cin, cout)
    assert int((b[0, 1:] == b[0, :-1]).sum()) > 0, "no split without live items"


@pytest.mark.parametrize("cin,cout", [(16, 16), (32, 64), (64, 128), (128, 128)])
def test_pass_live_only_in_last_chunk_of_split(cin, cout):
    """Offset 13 alone has neighbours, in a third as many tiles as there are splits: each split that gets an item then
    holds a single live chunk, its last, after chunks with no live item -- the pass's accumulator is first written by a
    split's last chunk."""
    n_in, n_out, kvol = 3000, 30011, 27
    rows = _chunk_rows(cout)
    splits = _row_splits(None, n_out, kvol, cin, cout).shape[1] - 1
    tiles = np.linspace(1, (n_out + 127) // 128 - 2, max(1, splits // 3)).astype(np.int64)
    nbr = _table(n_in, n_out, kvol, lambda k, r: (k == 13) & np.isin(r // 128, tiles), seed=2, density=0.5)
    masks = _check_live(nbr, n_in, cin, cout, 12, f"pass in last chunks {cin}->{cout}")
    opp = 128 // max(cin, 16)
    p13 = 13 // opp
    ppc = min((kvol + opp - 1) // opp, 512 // (64 if cout <= 64 else 128))
    live = _live_chunks(masks, n_out, rows, p13 * opp, opp)
    b = _row_splits(masks, n_out, kvol, cin, cout)
    hits = 0
    for r0, r1 in zip(b[p13 // ppc, :-1], b[p13 // ppc, 1:]):
        c0, c1 = r0 // rows, (r1 + rows - 1) // rows
        hits += int(c1 - c0 > 1 and live[c1 - 1] and not live[c0:c1 - 1].any())
    assert hits > 0, "no split has the pass live in its last chunk only"


@pytest.mark.parametrize("cin,cout", [(16, 64), (32, 32), (64, 64), (64, 128), (128, 64), (128, 128)])
def test_one_live_pass_per_chunk(cin, cout):
    """Exactly one live pass per 128-row tile, rotating, with runs of empty tiles: the dy ring must drain instead of
    waiting on a chunk whose items are not signalled yet."""
    n_in, n_out, kvol = 4000, 50000, 27
    opp = 128 // max(cin, 16)
    npass = (kvol + opp - 1) // opp

    def live(k, r):
        t = r // 128
        return (t % 5 != 3) & ((k // opp) == (t * 7) % npass)
    nbr = _table(n_in, n_out, kvol, live, seed=3, density=0.5)
    _check_live(nbr, n_in, cin, cout, 13, f"one pass per chunk {cin}->{cout}")


@pytest.mark.parametrize("cin,cout", [(16, 16), (64, 128)])
def test_null_masks_and_empty_table(cin, cout):
    """NULL masks: every item live, so the splits hold equal chunk counts (+-1); a table with no neighbour at all gives
    dw = 0 with masks."""
    ops = _ops()
    n_in, n_out, kvol = 2000, 9000, 27
    nbr = _table(n_in, n_out, kvol, lambda k, r: (k + r // 128) % 3 == 0, seed=4)
    _check_live(nbr, n_in, cin, cout, 14, f"mixed {cin}->{cout}")
    rows = _chunk_rows(cout)
    b = _row_splits(None, n_out, kvol, cin, cout)
    sizes = np.diff((b + rows - 1) // rows, axis=1)
    assert sizes.max() - sizes.min() <= 1, sizes
    empty = torch.full((kvol, n_out), -1, dtype=torch.int32, device=DEV)
    x, xb, dy, dyb = _operands(n_in, n_out, cin, cout, 15)
    dw = _wgrad(x, xb, empty, n_out, kvol, dy, dyb, cout, ops.table_tile_masks(empty))
    assert not bool(dw.any())


# (geometry, cin, cout) of every convolution of VoxelResBackBone8x (conv_input's 4-5 channels are padded to 16)
BACKBONE_WGRAD = [("L1", 5, 16), ("L1", 16, 16), ("down12", 16, 32), ("L2", 32, 32), ("down23", 32, 64), ("L3", 64, 64),
                  ("down34", 64, 128), ("L4", 128, 128), ("out", 128, 128)]


@pytest.mark.parametrize("geo_name,cin,cout", BACKBONE_WGRAD)
def test_backbone_wgrad_shapes_vs_fp64(full, geo_name, cin, cout):  # noqa: F811
    """Every wgrad shape of the backbone on full-size frames, with the rulebook's masks (twice: bit-identical) and with
    NULL masks, against the float64 reference of tests/test_gpu_layers.py (bf16-representable operands: rtol 1e-4)."""
    ops = _ops()
    geo = full[geo_name]
    rb = geo.rb
    x, w, _ = TL.make_operands(geo, cin, cout, "bf16", seed=cin * 100 + cout)
    dy = TL.bf16_round(torch.randn((geo.n_out, cout), device=DEV, generator=torch.Generator(device=DEV).manual_seed(cout)))
    cp = max(cin, 16)
    xp = torch.nn.functional.pad(x, (0, cp - cin)) if cp != cin else x
    assert rb.tile_masks is not None
    with_masks = _wgrad(xp, xp.to(torch.bfloat16), rb.nbr_fwd, rb.n_out, rb.kvol, dy, dy.to(torch.bfloat16), cout,
                        rb.tile_masks)
    again = _wgrad(xp, xp.to(torch.bfloat16), rb.nbr_fwd, rb.n_out, rb.kvol, dy, dy.to(torch.bfloat16), cout, rb.tile_masks)
    without = _wgrad(xp, xp.to(torch.bfloat16), rb.nbr_fwd, rb.n_out, rb.kvol, dy, dy.to(torch.bfloat16), cout, None)
    assert torch.equal(with_masks, again), geo_name
    _, dw_ref = TL.ref_conv_grads(x.double(), w.double(), geo, torch.zeros((geo.n_out, cout), dtype=torch.float64,
                                                                           device=DEV), dy.double())
    TL.check(with_masks[:, :, :cin].reshape(dw_ref.shape), dw_ref, what=f"{geo_name} wgrad {cin}->{cout}")
    TL.check(without[:, :, :cin].reshape(dw_ref.shape), dw_ref, what=f"{geo_name} wgrad {cin}->{cout} (NULL masks)")


# ------------------------------------------------------------------------------------------------ bias gradient
@pytest.mark.parametrize("training", [True, False])
@pytest.mark.parametrize("c", [6, 12, 16, 64, 128])
def test_bias_grad_from_bn_backward_vs_fp64_sum(c, training):
    """dbias of the BatchNorm backward pass = float64 sum of the fp32 dy the same pass wrote (vector and scalar kernels,
    training and eval gradient), run-to-run bit-identical."""
    ops = _ops()
    n = 70001
    g = torch.Generator(device=DEV).manual_seed(c)
    y = torch.randn((n, c), device=DEV, generator=g) * 2 + 0.5
    mean, rstd = y.mean(0), torch.rsqrt(y.var(0, unbiased=False) + 1e-3)
    gamma = torch.rand((c,), device=DEV, generator=g) + 0.5
    a = torch.relu((y - mean) * rstd * gamma)
    da = torch.randn((n, c), device=DEV, generator=g)

    def run():
        return ops._run_phases(ops._bn_backward_phases(da, y, a, gamma, mean, rstd, training, True, False, True, None, True),
                               None)
    dy, dyb, _, _, _, db = run()
    db2 = run()[5]
    assert torch.equal(db, db2)
    ref = dy.double().sum(0)
    err = (db.double() - ref).abs()
    # fp64 sums of fp32 values, reordered, then rounded to fp32: one fp32 rounding of the result
    bound = 2.0 ** -23 * ref.abs() + 1e-12 * dy.double().abs().sum(0)
    assert bool((err <= bound).all()), float((err / bound).max())


@pytest.mark.parametrize("prec", ["fp32", "bf16", "bf16x3"])
def test_bias_grad_fused_equals_stepwise(prec):
    """The fused layer backward (toda_layer_bwd) and the stepwise calls give the same bias gradient, bit for bit, and it
    is the rounding residue sum(dy) ~ 0 of a bias followed by training-mode BatchNorm."""
    ops = _ops()
    geo = TL.small_geo(20000, 31)
    cin, cout = 16, 32
    p = TL._prec(prec)
    x, w, b = TL.make_operands(geo, cin, cout, prec, seed=5)
    gout = torch.randn((geo.n_out, cout), device=DEV, generator=torch.Generator(device=DEV).manual_seed(6))

    def run(stepwise):
        bn = TL.make_bn(cout, 0.1, 4)
        if stepwise:
            ops.profile_begin()
        try:
            _, _, saved = ops._layer_forward(x, None, w, b, geo.rb, p, bn.weight, bn.bias, bn.running_mean, bn.running_var,
                                             bn.eps, bn.momentum, True, None, True, False)
            back = ops._layer_backward(gout, saved, geo.rb, p, True, True, False, True, True, True)
        finally:
            if stepwise:
                ops.profile_end()
        return back
    fused, step = run(False), run(True)
    for i, nm in enumerate(["dx", "dw", "db", "dgamma", "dbeta"]):
        assert torch.equal(fused[i], step[i]), nm
    assert float(fused[2].abs().max()) < 1e-3 * float(gout.abs().sum(0).max())
