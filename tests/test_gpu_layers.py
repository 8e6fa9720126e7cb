"""Layer-level parity of the product path against a float64 reference on the GPU.

What is checked, one layer at a time:
  A. ops.sparse_conv (forward, dgrad, wgrad, bias gradient) at full size: two nuScenes-shaped frames, every conv geometry
     of VoxelResBackBone8x (SubM at every level, the three stride-2 convs whose dgrad runs the parity-sorted path with
     out_rows, the (3,1,1)/(2,1,1) conv_out);
  B. the fused layer ops.conv_bn_act (toda_layer_fwd / toda_layer_bwd) in train mode, in eval mode under no_grad (the fused
     eval path) and in eval mode with an input gradient (the stepwise eval path); ragged sizes, channel counts whose
     BatchNorm runs on the scalar kernels, momentum 0.5 with running statistics far from the batch's, conv biases that
     put a channel's |mean| / std at ~1 and ~100;
  C. the residual block (ops.res_block through the plugin's SparseBasicBlock, and the unfused block an unmodified pcdet
     builds from SubMConv3d, ATen BatchNorm1d and ReLU);
  D. empty batches, which must behave like torch: empty outputs, zero parameter gradients, running statistics unchanged
     and num_batches_tracked + 1.

Reference: plain torch in float64 on the GPU.  Geometry comes from the CPU oracle's rulebooks
(oracle.spconv_oracle.subm_rulebook / sparse_rulebook), never from the product's tables; convolution is
out.index_add_(0, out_rows, x[in_rows] @ W_k) over the offsets with autograd giving dgrad and wgrad; BatchNorm is
F.batch_norm on float64 copies of the running statistics; then residual and ReLU.  The ReLU of the reference is gated with
the product's mask (a > 0), so that a mask that flips at the kink is not counted as a kernel error; separately the masks
must agree wherever the reference's pre-activation exceeds 1e-5 of its scale.

Rounding model.  fp32 and bf16x3: the reference sees the same fp32 inputs.  bf16: x, the weights and the cotangent are
bf16-representable, and the reference rounds to bf16 exactly where the product does -- the conv's incoming gradient dy
(for dgrad when the dgrad runs on tensor cores, for wgrad when the wgrad does) and, inside a residual block, the hidden
activation that the second convolution reads.

Tolerances (PU.assert_close, rtol plus atol_scale x the largest reference magnitude):
  * fp32 and bf16x3, every output: rtol 1e-4, atol_scale 1e-5;
  * bf16, a single layer's forward: rtol 1e-4 (identical operands, only the fp32 accumulation order differs);
  * bf16, anything downstream of a rounding inside the product (every backward of a BatchNorm layer, the second conv of a
    residual block): rtol 1e-3, atol_scale 1e-4.  The product and the reference round values that differ by ~1e-6
    relative (~1e-4 with the statistics error at |mean| / std = 100); where that difference straddles a bf16 rounding
    boundary one term moves by one bf16 spacing.  Measured, such a flip of a large term in a small dgrad sum reaches
    2.5-10x that bound, so dx and dw also get an explicit allowance for every term that can flip (RefLayer.backward).
    The ReLU masks after the second conv of a block are compared clear of 1e-3 of the scale, the forward tolerance there.
  * bf16x3 dx and dw: plus 2^-15 of the absolute sum of the terms (the split's dropped lo*lo term and residues).
    Measured: wgrad of a block's second conv over 2.7e5 rows of a non-negative (ReLU) operand, where the result cancels,
    reaches 1.6x rtol 1e-4 without it.
  * the gradient of a conv bias in front of a training-mode BatchNorm is zero up to rounding: it is bounded by rtol x the
    per-channel sum of |dy| instead.

Limit of the epilogue statistics (bf16 and bf16x3 training): the tensor-core kernels accumulate the per-channel sums of y
and y^2 in fp32 per warp and tile, and the variance is E[y^2] - E[y]^2.  A CPU emulation of that arithmetic gives rstd
errors of 4e-6 to 3e-5 at |mean| / std = 100 for 2e4-5e5 rows, but 1.7e-4 at ratio 300, and ~4e-4 at ratio 100 over only
~130 rows (the fp32 error of a 32-row warp sum of y^2 is not averaged down).  The ratio-100 channels therefore run on the
1e5-row SubM level only (measured there: a, running_var and dx within 0.6-1.0 of rtol 1e-4); on the 2.9e4-row conv_out
level ratio 100 took dx to 1.1x the bound in bf16x3, since BatchNorm backward roughly doubles the rstd error.  The ragged
sizes run at ratio ~1.
"""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from tests import parity_utils as PU

pytestmark = pytest.mark.gpu
DEV = "cuda"
PRECISIONS = ("fp32", "bf16", "bf16x3")


# ---------------------------------------------------------------------------------------------- helpers
def _ops():
    from toda_b200 import ops
    return ops


def _prec(name):
    ops = _ops()
    return {"fp32": ops.CONV_FP32, "bf16": ops.CONV_BF16, "bf16x3": ops.CONV_BF16X3}[name]


def bf16_round(t):
    return t.to(torch.bfloat16).to(t.dtype)


def check(got, want, rtol=PU.RTOL, atol_scale=1e-5, what="", allow=None):
    """PU.assert_close, after printing the measured maximum error (absolute, and as a fraction of the bound).  allow: an
    element-wise allowance added to the bound (the rounding error model of RefLayer.backward)."""
    a = got.detach().double().cpu().numpy() if torch.is_tensor(got) else np.asarray(got, np.float64)
    b = want.detach().double().cpu().numpy() if torch.is_tensor(want) else np.asarray(want, np.float64)
    extra = allow.detach().double().cpu().numpy() if allow is not None else 0.0
    if a.size and a.shape == b.shape:
        scale = max(float(np.abs(b).max()), 1e-30)
        err = np.abs(a - b)
        frac = float((err / (rtol * np.abs(b) + atol_scale * scale + extra)).max())
        print(f"{what}: max err {err.max():.3e} at scale {scale:.3e} ({frac:.2f} of the bound rtol={rtol:g} "
              f"atol_scale={atol_scale:g}{' + rounding allowance' if allow is not None else ''})")
        if allow is not None:
            assert frac <= 1.0, f"{what}: max err {err.max():.3e} is {frac:.2f} of the bound"
    PU.assert_close(a, b, rtol=rtol, atol_scale=atol_scale + (float(np.max(extra)) / scale if allow is not None and a.size else 0.0),
                    what=what)


def check_zero_bias_grad(got, dy_ref, rtol, what):
    """Conv bias in front of a training-mode BatchNorm: the gradient is sum(dy) = 0 up to rounding; bound it by rtol x the
    per-channel sum of |dy|."""
    g = got.detach().double()
    bound = rtol * dy_ref.abs().sum(0)
    frac = float((g.abs() / bound.clamp_min(1e-300)).max()) if g.numel() else 0.0
    print(f"{what}: max |db| {float(g.abs().max()) if g.numel() else 0.0:.3e} ({frac:.2f} of rtol x sum|dy|)")
    assert bool((g.abs() <= bound).all()), (what, frac)


def check_masks(mask, z_ref, what, kink=1e-5):
    """The product's ReLU mask agrees with the reference's sign wherever the pre-activation is clear of the kink (|z| above
    `kink` x its scale: 1e-5, or the forward tolerance 1e-3 downstream of a bf16 rounding inside the product)."""
    z = z_ref.detach()
    if z.numel() == 0:
        return
    clear = z.abs() > kink * z.abs().max()
    bad = int(((mask > 0) != (z > 0))[clear].sum())
    print(f"{what}: {bad} mask disagreements clear of the kink, {int((~clear).sum())} elements at the kink")
    assert bad == 0, (what, bad)


class Geo:
    """One conv geometry: the product's rulebook and the oracle's pairs (as GPU index tensors)."""

    def __init__(self, rb, pairs, n_in, n_out, ksize):
        self.rb, self.n_in, self.n_out, self.ksize = rb, n_in, n_out, list(ksize)
        self.pairs = [(torch.from_numpy(np.asarray(i, np.int64)).to(DEV), torch.from_numpy(np.asarray(o, np.int64)).to(DEV))
                      for i, o in pairs]


def ref_conv(x, w, geo):
    """sum over offsets k of out.index_add_(0, out_rows, x[in_rows] @ W_k); w is the (Cout, kz, ky, kx, Cin) parameter."""
    cout, cin = w.shape[0], w.shape[4]
    wk = w.reshape(cout, -1, cin)
    out = x.new_zeros((geo.n_out, cout))
    for k, (i, o) in enumerate(geo.pairs):
        if i.numel():
            out = out.index_add(0, o, x[i] @ wk[:, k, :].t())
    return out


def _subm_geo(index, coords_np, shape):
    from oracle import spconv_oracle as S
    ops = _ops()
    rb = ops.rulebook_subm(index, [3, 3, 3])
    assert np.array_equal(rb.out_coords.cpu().numpy(), coords_np)        # canonical input: SubM keeps the rows
    return Geo(rb, S.subm_rulebook(coords_np, shape, [3, 3, 3]), rb.n_in, rb.n_out, [3, 3, 3])


def _sparse_geo(index, coords_np, shape, k, s, p, tag):
    from oracle import spconv_oracle as S
    ops = _ops()
    rb, index_out = ops.rulebook_sparse(index, k, s, p, tag)
    oi, oshape, pairs = S.sparse_rulebook(coords_np, shape, k, s, p)
    assert list(oshape) == list(rb.out_shape)
    assert np.array_equal(rb.out_coords.cpu().numpy(), oi)
    return Geo(rb, pairs, rb.n_in, rb.n_out, k), index_out, oi, list(oshape)


@pytest.fixture(scope="module")
def full():
    """Two full-size nuScenes-shaped frames (voxelized as the plan-kernel chain test does) and every conv geometry of
    VoxelResBackBone8x on them.  Keys: 'L1'..'L4' (SubM at each level), 'down12', 'down23', 'down34', 'out'."""
    from toda_b200 import synth
    ops = _ops()
    cfg = synth.CONFIGS["nus_0075"]
    frames, collated = synth.make_batch("nus_0075", 2)
    dev = torch.device(DEV, 0)
    offs = torch.from_numpy(np.cumsum([0] + [f.shape[0] for f in frames]).astype(np.int32)).to(dev)
    grid = synth.grid_size_xyz(cfg["pc_range"], cfg["voxel_size"])
    _, coords, _, _ = ops.voxelize(torch.from_numpy(collated).to(dev), offs, cfg["pc_range"], cfg["voxel_size"], 10, 120000,
                                   xyz_col=1, feat_col=1, num_features=5, order=ops.ORDER_CANONICAL, grid=grid)
    shape = [int(grid[2]) + 1, int(grid[1]), int(grid[0])]
    index = ops.OccupancyIndex(2, shape, dev, "layers")
    index.insert(coords)
    index.build(coords.shape[0], known_n=coords.shape[0])
    c = coords.cpu().numpy()
    geos = {}
    down = [((3, 3, 3), (2, 2, 2), (1, 1, 1)), ((3, 3, 3), (2, 2, 2), (1, 1, 1)), ((3, 3, 3), (2, 2, 2), (0, 1, 1))]
    for lvl in range(1, 5):
        geos[f"L{lvl}"] = _subm_geo(index, c, shape)
        if lvl < 4:
            k, s, p = down[lvl - 1]
            geos[f"down{lvl}{lvl + 1}"], index, c, shape = _sparse_geo(index, c, shape, list(k), list(s), list(p), ("layers", lvl))
    geos["out"], _, _, _ = _sparse_geo(index, c, shape, [3, 1, 1], [2, 1, 1], [0, 0, 0], ("layers", 5))
    print("full-size rows per level: " + ", ".join(f"{k} {g.n_in}->{g.n_out}" for k, g in geos.items()))
    yield geos


def small_geo(n, seed):
    """SubM 3x3x3 over n random voxels of one frame (canonical order): ragged row counts."""
    ops = _ops()
    shape = [40, 50, 60]
    _, idx = PU.random_sparse(seed, 1, shape, n, 1)
    index = ops.OccupancyIndex(1, shape, torch.device(DEV, 0), "layers_small")
    index.insert(torch.from_numpy(idx).to(DEV))
    index.build(n, known_n=n)
    return _subm_geo(index, idx, shape)


def make_operands(geo, cin, cout, prec, seed, bias=True, wscale=None):
    """x, weight (Cout, k..., Cin), bias: fp32; bf16-representable in bf16 mode."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    kvol = geo.ksize[0] * geo.ksize[1] * geo.ksize[2]
    wscale = (1.0 / np.sqrt(kvol * cin)) if wscale is None else wscale
    x = torch.randn((geo.n_in, cin), device=DEV, generator=g)
    w = torch.randn((cout, *geo.ksize, cin), device=DEV, generator=g) * wscale
    b = torch.randn((cout,), device=DEV, generator=g) * 0.1 if bias else None
    if prec == "bf16":
        x, w = bf16_round(x), bf16_round(w)
    return x, w, b


def _uses_tc(cin, cout, kvol, prec):
    from toda_b200 import _C
    L = _C.lib()
    return bool(L.toda_spconv_uses_tensor_cores(cin, cout, kvol, _prec(prec))), \
        bool(L.toda_spconv_wgrad_uses_tensor_cores(cin, cout, kvol, _prec(prec)))


def _rounders(cin, cout, kvol, prec):
    """bf16 rounding of the conv's incoming gradient for (dgrad, wgrad), where the product's kernels read its bf16 copy."""
    ident = lambda t: t  # noqa: E731
    if prec != "bf16":
        return ident, ident
    dgrad_tc, _ = _uses_tc(cout, cin, kvol, prec)
    _, wgrad_tc = _uses_tc(cin, cout, kvol, prec)
    return (bf16_round if dgrad_tc else ident), (bf16_round if wgrad_tc else ident)


def bf16_flip_ulp(v, rel, abs_tol=0.0):
    """bf16 spacing at |v| where v lies within rel x |v| + abs_tol of a round-to-nearest midpoint (a value the product,
    computing v with that difference, may round to the other neighbour), else 0."""
    a = v.abs()
    ulp = torch.exp2(torch.floor(torch.log2(a.clamp_min(1e-300))) - 7)
    frac = a / ulp - torch.floor(a / ulp)
    near = ((frac - 0.5).abs() * ulp <= rel * a + abs_tol) & (a > 0)
    return torch.where(near, ulp, torch.zeros_like(a))


def ref_conv_grads(x, w, geo, cot_x, cot_w):
    """(dgrad of cot_x, wgrad of cot_w) of ref_conv at (x, w)."""
    xl, wl = x.detach().requires_grad_(True), w.detach().requires_grad_(True)
    y = ref_conv(xl, wl, geo)
    dx, = torch.autograd.grad(y, [xl], cot_x, retain_graph=True)
    dw, = torch.autograd.grad(y, [wl], cot_w)
    return dx, dw


# The product's dy (BatchNorm backward, fp32) differs from the reference's by up to ~2x the relative error of its batch
# statistics (rstd up to ~3e-5 from the epilogue sums at |mean| / std = 100, see above) plus a few fp32 roundings.
DY_REL = 1e-4
# bf16x3 products: hi*hi + hi*lo + lo*hi of the split operands; the dropped lo*lo term and the residues of the splits leave
# at most ~2^-15 of |x| |dy| per term.
X3_REL = 2.0 ** -15


class RefLayer:
    """float64 conv (+ bias) -> F.batch_norm (+ residual) -> ReLU gated by the product's mask, with its own backward."""

    def __init__(self, x, w, b, geo, bn, training, residual=None, mask=None):
        self.geo = geo
        self.x = x.detach().double().requires_grad_(True)
        self.w = w.detach().double().requires_grad_(True)
        self.yc = ref_conv(self.x, self.w, geo)
        self.y = (self.yc.detach() + (b.detach().double() if b is not None else 0.0)).requires_grad_(True)
        self.gamma = bn.weight.detach().double().requires_grad_(True)
        self.beta = bn.bias.detach().double().requires_grad_(True)
        self.running_mean = bn.running_mean.detach().double().clone()
        self.running_var = bn.running_var.detach().double().clone()
        self.training = training
        yd = self.y.detach()
        mean, var = (yd.mean(0), yd.var(0, unbiased=False)) if training else (self.running_mean.clone(), self.running_var.clone())
        self.var_eps = var + bn.eps
        self.rstd = self.var_eps.rsqrt()
        self.xhat = (yd - mean) * self.rstd
        self.fy = None           # allowance on y (fwd_allowance)
        self.h_allow = self.out_allow = None      # allowances on the conv input and on the output (residual blocks)
        self.res = residual.detach().double().requires_grad_(True) if residual is not None else None
        self.z = F.batch_norm(self.y, self.running_mean, self.running_var, self.gamma, self.beta, training, bn.momentum, bn.eps)
        if self.res is not None:
            self.z = self.z + self.res
        self.mask = mask.double() if mask is not None else torch.ones_like(self.z)
        self.a = self.z.detach() * self.mask

    def fwd_allowance(self, u_in):
        """Allowance on this layer's output when its conv input may differ from the reference's by u_in per element (bf16
        rounding flips of the input, see bf16_flip_ulp): |W| propagates it to y, BatchNorm scales it by |gamma| rstd and, in
        training, adds the shift of the batch mean and the relative change of the batch variance."""
        fy = ref_conv(u_in, self.w.detach().abs(), self.geo)
        gr = self.gamma.detach().abs() * self.rstd
        if self.training:
            dvar = 2 * ((self.xhat.abs() / self.rstd) * fy).mean(0)
            fz = gr * (fy + fy.mean(0)) + self.gamma.detach().abs() * self.xhat.abs() * dvar / (2 * self.var_eps)
        else:
            fz = gr * fy
        self.fy = fy
        return fz * self.mask

    def backward(self, da, prec, round_d, round_w, da_allow=None, x_allow=None):
        """-> dict dx, dw, db, dgamma, dbeta, dres, dy, and the rounding allowances fdx, fdw, fdgamma, fdbeta.  round_d /
        round_w: the rounding of dy seen by dgrad / wgrad.  x_allow: allowance on the conv's input (as for fwd_allowance).
        da_allow: allowance on da from rounding flips upstream (a residual block's second dgrad).  Those flips are
        independent and of either sign, so they are carried root-sum-square, 3 sigma, through BatchNorm and this conv.

        Error model of the allowances.  bf16: where dy lies within DY_REL of a bf16 rounding midpoint the product may round
        it to the other neighbour, one bf16 spacing u away; such a flip moves dx by u |W_k| and dw by u |x| -- up to 5-10x
        the rtol 1e-3 / atol_scale 1e-4 bound when a large term of a small sum flips.  The allowance is the reference
        dgrad / wgrad of |x|, |W| and those u (zero elsewhere).  bf16x3: X3_REL |dy| per term, through |x|, |W|."""
        gz = da.double() * self.mask
        dy, dgamma, dbeta = torch.autograd.grad(self.z, [self.y, self.gamma, self.beta], gz, retain_graph=True)
        dx, = torch.autograd.grad(self.yc, [self.x], round_d(dy), retain_graph=True)
        dw, = torch.autograd.grad(self.yc, [self.w], round_w(dy))
        # allowance on dy: from y (the xhat term of the training-mode backward), and (root-sum-square) from da
        gr = self.gamma.detach().abs() * self.rstd
        ga = da_allow.double() * self.mask if da_allow is not None else torch.zeros_like(dy)
        n = max(dy.shape[0], 1)
        var_dy = (gr * ga) ** 2
        if self.training:
            var_dy = var_dy + gr ** 2 * ((ga ** 2).sum(0) / n ** 2 + self.xhat ** 2 * ((ga * self.xhat) ** 2).sum(0) / n ** 2)
        sd_dy = 3 * var_dy.sqrt()
        fdy = torch.zeros_like(dy)
        if self.training and self.fy is not None:
            fdy = gr * self.rstd * (self.fy + self.fy.mean(0)) * (gz * self.xhat).mean(0).abs()
        if prec == "bf16":
            u = bf16_flip_ulp(dy, DY_REL, fdy + sd_dy)
            ud, uw = fdy + (u if round_d is bf16_round else 0 * u), fdy + (u if round_w is bf16_round else 0 * u)
        else:
            ud = uw = fdy + (X3_REL * dy.abs() if prec == "bf16x3" else 0 * dy)
        fdx, fdw = ref_conv_grads(self.x.abs(), self.w.abs(), self.geo, ud, uw)
        if x_allow is not None:
            fdw = fdw + ref_conv_grads(x_allow, self.w.abs(), self.geo, torch.zeros_like(dy), round_w(dy).abs() + uw)[1]
        if da_allow is not None:
            vdx, vdw = ref_conv_grads(self.x.detach() ** 2, self.w.detach() ** 2, self.geo, sd_dy ** 2, sd_dy ** 2)
            fdx, fdw = fdx + vdx.sqrt(), fdw + vdw.sqrt()
        return dict(dx=dx, dw=dw, db=dy.sum(0), dgamma=dgamma, dbeta=dbeta, dres=gz if self.res is not None else None, dy=dy,
                    fdx=fdx, fdw=fdw, fdgamma=3 * ((ga * self.xhat) ** 2).sum(0).sqrt(), fdbeta=3 * (ga ** 2).sum(0).sqrt())


def make_bn(c, momentum, seed, rv_init=None, y_ref=None):
    """BatchNorm1d(eps=1e-3) on the GPU with random affine parameters.  Running statistics: rv_init (a constant, e.g. far
    below the batch variance), or random values around the batch's statistics of y_ref (eval cases)."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    bn = torch.nn.BatchNorm1d(c, eps=1e-3, momentum=momentum).to(DEV)
    with torch.no_grad():
        bn.weight.copy_(torch.rand((c,), device=DEV, generator=g) + 0.5)
        bn.bias.copy_(torch.rand((c,), device=DEV, generator=g) - 0.5)
        if y_ref is not None and y_ref.shape[0] > 1:
            m, s = y_ref.mean(0).float(), y_ref.std(0).float()
            bn.running_mean.copy_(m + 0.3 * s * torch.randn((c,), device=DEV, generator=g))
            bn.running_var.copy_(s * s * (torch.rand((c,), device=DEV, generator=g) * 1.5 + 0.5))
        else:
            bn.running_mean.copy_(torch.randn((c,), device=DEV, generator=g) * 0.2)
            bn.running_var.copy_(torch.rand((c,), device=DEV, generator=g) * 1.5 + 0.5)
        if rv_init is not None:
            bn.running_var.fill_(rv_init)
    return bn


def offset_bias(x, w, geo, ratios):
    """Conv bias that puts channel c's |mean| / std of y at ratios[c % len(ratios)] (from a bias-free reference pass)."""
    yc = ref_conv(x.double(), w.double(), geo)
    m, s = yc.mean(0), yc.std(0)
    r = torch.tensor([ratios[c % len(ratios)] for c in range(w.shape[0])], dtype=torch.float64, device=DEV)
    return (r * s - m).float()


def bwd_tols(prec):
    return (1e-3, 1e-4) if prec == "bf16" else (PU.RTOL, 1e-5)


# ---------------------------------------------------------------------------------------------- A. convolutions at scale
CONV_CASES = [("L1", 5, 16), ("L1", 16, 16), ("L2", 32, 32), ("L3", 64, 64), ("L4", 128, 128),
              ("down12", 16, 32), ("down23", 32, 64), ("down34", 64, 128), ("out", 128, 128)]


@pytest.mark.parametrize("prec", PRECISIONS)
@pytest.mark.parametrize("geo_name,cin,cout", CONV_CASES)
def test_sparse_conv_at_scale_vs_fp64(full, geo_name, cin, cout, prec):
    """ops.sparse_conv forward, dgrad, wgrad and bias gradient on full-size geometry (SubM levels: >= 4 tiles of 128 rows
    per CTA; strided dgrad: parity-sorted rows scattered back through out_rows) against the fp64 reference.  The conv's
    operands are exact in every precision (bf16: bf16-representable x, w and cotangent), so rtol 1e-4 throughout."""
    ops = _ops()
    geo = full[geo_name]
    x, w, b = make_operands(geo, cin, cout, prec, seed=cin * 1000 + cout)
    g = torch.randn((geo.n_out, cout), device=DEV, generator=torch.Generator(device=DEV).manual_seed(7))
    if prec == "bf16":
        g = bf16_round(g)
    xx, ww, bb = x.clone().requires_grad_(True), w.clone().requires_grad_(True), b.clone().requires_grad_(True)
    y = ops.sparse_conv(xx, ww, bb, geo.rb, _prec(prec))
    y.backward(g)
    xr, wr = x.double().requires_grad_(True), w.double().requires_grad_(True)
    yr = ref_conv(xr, wr, geo) + b.double()
    yr.backward(g.double())
    tag = f"{geo_name} {cin}->{cout} {prec} n={geo.n_in}->{geo.n_out}"
    check(y, yr, what=f"conv fwd {tag}")
    check(xx.grad, xr.grad, what=f"conv dgrad {tag}")
    check(ww.grad, wr.grad, what=f"conv wgrad {tag}")
    check(bb.grad, g.double().sum(0), what=f"conv bias grad {tag}")


# ---------------------------------------------------------------------------------------------- B. fused layer
# name -> (geometry, cin, cout, momentum, running_var start (None: random), |mean|/std of y per channel (None: no conv
# bias, as in the backbones' conv + BN layers; without a bias gradient to compute, the bf16 backward skips the fp32 dy))
LAYER_CASES = {
    "input_5_16": ("L1", 5, 16, 0.01, None, None),
    "subm_64_offsets": ("L3", 64, 64, 0.5, 1e-3, (1.0, 100.0)),
    "down_32_64": ("down23", 32, 64, 0.5, 1e-3, None),
    "out_128": ("out", 128, 128, 0.5, None, (1.0,)),
}


def run_layer_case(geo, cin, cout, prec, mode, momentum, rv_init, ratios, seed, tag):
    """ops.conv_bn_act (ReLU) on `geo` against RefLayer.  mode: 'train', 'eval_nograd' (fused eval path) or 'eval_grad'
    (stepwise eval path)."""
    ops = _ops()
    x, w, _ = make_operands(geo, cin, cout, prec, seed, bias=False)
    b = offset_bias(x, w, geo, ratios) if ratios is not None else None
    training = mode == "train"
    y0 = ref_conv(x.double(), w.double(), geo) + (b.double() if b is not None else 0.0) if not training else None
    bn = make_bn(cout, momentum, seed + 1, rv_init=rv_init if training else None, y_ref=y0)
    bn.train(training)
    nbt0 = int(bn.num_batches_tracked)
    rm0, rv0 = bn.running_mean.clone(), bn.running_var.clone()
    g = torch.randn((geo.n_out, cout), device=DEV, generator=torch.Generator(device=DEV).manual_seed(seed + 2))
    ref_bn = torch.nn.BatchNorm1d(cout, eps=bn.eps, momentum=bn.momentum).to(DEV)
    ref_bn.load_state_dict(bn.state_dict())
    bf16 = prec == "bf16"
    if mode == "eval_nograd":
        with torch.no_grad():
            a, ab = ops.conv_bn_act(x, w, b, geo.rb, _prec(prec), bn, None, True, None, bf16)
    else:
        xx, ww = x.clone().requires_grad_(True), w.clone().requires_grad_(True)
        bb = b.clone().requires_grad_(True) if b is not None else None
        a, ab = ops.conv_bn_act(xx, ww, bb, geo.rb, _prec(prec), bn, None, True, None, bf16)
        a.backward(g)
    if bf16:
        assert torch.equal(ab, a.detach().to(torch.bfloat16))
    ref = RefLayer(x, w, b, geo, ref_bn, training, mask=(a.detach() > 0))
    check_masks(a.detach(), ref.z, f"layer mask {tag}")
    check(a, ref.a, what=f"layer a {tag}")
    if training:
        check(bn.running_mean, ref.running_mean, what=f"layer running_mean {tag}")
        check(bn.running_var, ref.running_var, what=f"layer running_var {tag}")
        assert int(bn.num_batches_tracked) == nbt0 + 1
    else:
        assert torch.equal(bn.running_mean, rm0) and torch.equal(bn.running_var, rv0)
        assert int(bn.num_batches_tracked) == nbt0
    if mode == "eval_nograd":
        return
    kvol = geo.ksize[0] * geo.ksize[1] * geo.ksize[2]
    rd, rw = _rounders(cin, cout, kvol, prec)
    r = ref.backward(g, prec, rd, rw)
    rtol, atol = bwd_tols(prec)
    check(xx.grad, r["dx"], rtol, atol, what=f"layer dx {tag}", allow=r["fdx"])
    check(ww.grad, r["dw"], rtol, atol, what=f"layer dw {tag}", allow=r["fdw"])
    check(bn.weight.grad, r["dgamma"], rtol, atol, what=f"layer dgamma {tag}")
    check(bn.bias.grad, r["dbeta"], rtol, atol, what=f"layer dbeta {tag}")
    if bb is None:
        return
    if training:
        check_zero_bias_grad(bb.grad, r["dy"], rtol, what=f"layer db {tag}")
    else:
        check(bb.grad, r["db"], rtol, atol, what=f"layer db {tag}")


@pytest.mark.parametrize("prec", PRECISIONS)
@pytest.mark.parametrize("mode", ["train", "eval_nograd", "eval_grad"])
@pytest.mark.parametrize("case", list(LAYER_CASES))
def test_conv_bn_act_full_size_vs_fp64(full, case, mode, prec):
    """Fused conv -> BatchNorm1d -> ReLU on full-size geometry: outputs, every gradient and the running statistics.  In
    bf16 / bf16x3 training the statistics come from the conv epilogue (toda_bn_apply_sums)."""
    geo_name, cin, cout, momentum, rv_init, ratios = LAYER_CASES[case]
    run_layer_case(full[geo_name], cin, cout, prec, mode, momentum, rv_init, ratios, seed=100 * list(LAYER_CASES).index(case),
                   tag=f"{case} {mode} {prec}")


@pytest.mark.parametrize("prec", PRECISIONS)
@pytest.mark.parametrize("mode", ["train", "eval_nograd", "eval_grad"])
@pytest.mark.parametrize("n", [1, 127, 129])
@pytest.mark.parametrize("cin,cout", [(64, 64), (16, 12), (16, 6)])
def test_conv_bn_act_ragged_vs_fp64(n, cin, cout, mode, prec):
    """Ragged row counts (a last tile of 1 row, one short of and one past a 128-row tile) and channel counts whose
    BatchNorm runs on the scalar kernels (12: C/4 does not divide the block; 6: not a multiple of 4) and whose convolution
    runs on the FFMA kernel in every precision.  n = 1 in eval mode only: torch refuses batch statistics over one row."""
    if n == 1 and mode == "train":
        pytest.skip("batch statistics over one row")
    run_layer_case(small_geo(n, seed=n), cin, cout, prec, mode, 0.5, 1e-3, None, seed=n + 1000 * cin + cout,
                   tag=f"ragged n={n} {cin}->{cout} {mode} {prec}")


# ---------------------------------------------------------------------------------------------- C. residual block
def _block(cin, prec, seed):
    """The plugin's SparseBasicBlock with random (bf16: representable) weights and random BatchNorm parameters."""
    import toda_b200.pcdet_plugin as P
    torch.manual_seed(seed)
    blk = P.SparseBasicBlock(cin, cin, indice_key="blk").to(DEV)
    with torch.no_grad():
        for conv in (blk.conv1, blk.conv2):
            if prec == "bf16":
                conv.weight.copy_(bf16_round(conv.weight))
        for bn in (blk.bn1, blk.bn2):
            bn.weight.uniform_(0.5, 1.5)
            bn.bias.uniform_(-0.5, 0.5)
            bn.running_mean.normal_(0.0, 0.2)
            bn.running_var.uniform_(0.5, 2.0)
            bn.momentum = 0.5
    return blk


def _bn_states(blk):
    return [{k: v.clone() for k, v in bn.state_dict().items()} for bn in (blk.bn1, blk.bn2)]


def _ref_block(blk, before, x, geo, training, h_prod, out_mask, prec):
    """Reference SparseBasicBlock (spconv_backbone.py L30-66): conv1-bn1-relu, conv2-bn2, + identity, relu, starting from
    the BatchNorm states `before` the product's step."""
    bn1 = torch.nn.BatchNorm1d(blk.bn1.num_features, eps=blk.bn1.eps, momentum=blk.bn1.momentum).to(DEV)
    bn2 = torch.nn.BatchNorm1d(blk.bn2.num_features, eps=blk.bn2.eps, momentum=blk.bn2.momentum).to(DEV)
    bn1.load_state_dict(before[0])
    bn2.load_state_dict(before[1])
    l1 = RefLayer(x, blk.conv1.weight, blk.conv1.bias, geo, bn1, training, mask=h_prod > 0)
    h_in = bf16_round(l1.a) if prec == "bf16" else l1.a
    l2 = RefLayer(h_in, blk.conv2.weight, blk.conv2.bias, geo, bn2, training, residual=x, mask=out_mask)
    # bf16: conv2 reads bf16(h) of the product's h, which agrees with the reference's to ~1e-6; where the two sit on either
    # side of a rounding midpoint conv2's inputs are one bf16 spacing apart.  Those flips are known exactly (the product's h
    # is saved for backward).  Measured without this allowance: the block output 2.2x its rtol 1e-3 / atol_scale 1e-4 bound.
    l2.h_allow = (bf16_round(h_prod.double()) - h_in).abs() if prec == "bf16" else None
    l2.out_allow = l2.fwd_allowance(l2.h_allow) if prec == "bf16" else None
    return l1, l2


def _block_backward(l1, l2, g, cin, prec):
    rd, rw = _rounders(cin, cin, 27, prec)
    r2 = l2.backward(g, prec, rd, rw, x_allow=l2.h_allow)
    r1 = l1.backward(r2["dx"], prec, rd, rw, da_allow=r2["fdx"])
    r1["dx"] = r1["dx"] + r2["dres"]
    return r1, r2


def _compare_block(blk, xx, out, h, l1, l2, r1, r2, training, prec, tag):
    bf16 = prec == "bf16"
    rtol, atol = bwd_tols(prec)
    check_masks(h, l1.z, f"block h mask {tag}")
    check_masks(out, l2.z, f"block out mask {tag}", kink=1e-3 if bf16 else 1e-5)
    check(h, l1.a, what=f"block h {tag}")
    # the second conv reads the bf16-rounded hidden activation: downstream of a rounding inside the product
    check(out, l2.a, *((rtol, atol) if bf16 else (PU.RTOL, 1e-5)), what=f"block out {tag}", allow=l2.out_allow)
    check(xx.grad, r1["dx"], rtol, atol, what=f"block dx {tag}", allow=r1["fdx"])
    for i, (conv, bn, r, l) in enumerate(((blk.conv1, blk.bn1, r1, l1), (blk.conv2, blk.bn2, r2, l2)), 1):
        check(conv.weight.grad, r["dw"], rtol, atol, what=f"block dw{i} {tag}", allow=r["fdw"])
        check(bn.weight.grad, r["dgamma"], rtol, atol, what=f"block dgamma{i} {tag}", allow=r["fdgamma"])
        check(bn.bias.grad, r["dbeta"], rtol, atol, what=f"block dbeta{i} {tag}", allow=r["fdbeta"])
        if training:
            check_zero_bias_grad(conv.bias.grad, r["dy"], rtol, what=f"block db{i} {tag}")
            check(bn.running_mean, l.running_mean, *((rtol, atol) if (bf16 and i == 2) else (PU.RTOL, 1e-5)),
                  what=f"block running_mean{i} {tag}")
            check(bn.running_var, l.running_var, *((rtol, atol) if (bf16 and i == 2) else (PU.RTOL, 1e-5)),
                  what=f"block running_var{i} {tag}")
        else:
            check(conv.bias.grad, r["db"], rtol, atol, what=f"block db{i} {tag}")


def _canonical_tensor(geo, cin, prec, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    x = torch.randn((geo.n_in, cin), device=DEV, generator=g)
    if prec == "bf16":
        x = bf16_round(x)
    return x, geo.rb.out_coords


@pytest.mark.parametrize("prec", PRECISIONS)
@pytest.mark.parametrize("mode", ["train", "eval_grad"])
@pytest.mark.parametrize("geo_name,c", [("L2", 32), ("L4", 128)])
def test_res_block_vs_fp64(full, geo_name, c, mode, prec):
    """The plugin's SparseBasicBlock (ops.res_block: both layers fused, the residual-branch gradient added in conv1's dgrad
    epilogue, the bf16 shadow of the hidden activation, the elided fp32 dy) against the reference block.  The product's
    hidden ReLU mask is read from the saved tensors of the block's autograd node."""
    from toda_b200.spconv_compat import pytorch as G
    geo = full[geo_name]
    training = mode == "train"
    blk = _block(c, prec, seed=c)
    blk.train(training)
    x, coords = _canonical_tensor(geo, c, prec, seed=c + 1)
    g = torch.randn((geo.n_out, c), device=DEV, generator=torch.Generator(device=DEV).manual_seed(c + 2))
    before = _bn_states(blk)
    G.set_conv_precision(prec)
    try:
        xx = x.clone().requires_grad_(True)
        st = G.SparseConvTensor(xx, coords, geo.rb.in_shape, 2).canonical(assume_canonical=True)
        out = blk(st).features
        h = out.grad_fn.saved_tensors[4]          # layer 1's activation (ops._ResBlock saves (x, xb, w, y, a, ...) per layer)
        out.backward(g)
    finally:
        G.set_conv_precision("fp32")
    l1, l2 = _ref_block(blk, before, x, geo, training, h.detach(), out.detach() > 0, prec)
    r1, r2 = _block_backward(l1, l2, g, c, prec)
    _compare_block(blk, xx, out.detach(), h.detach(), l1, l2, r1, r2, training, prec, f"{geo_name} {mode} {prec}")
    nbt = 1 if training else 0
    assert int(blk.bn1.num_batches_tracked) == nbt and int(blk.bn2.num_batches_tracked) == nbt


@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_unfused_res_block_vs_fp64(full, prec):
    """The block as an unmodified pcdet builds it (spconv_backbone.py L30-66): SubMConv3d, then ATen BatchNorm1d and ReLU
    through replace_feature, + identity.features.  In bf16 training the convolutions also accumulate epilogue BatchNorm
    sums; replace_feature must drop them, since ATen's BatchNorm computes its own."""
    from toda_b200.spconv_compat import pytorch as G
    geo, c = full["L2"], 32
    blk = _block(c, prec, seed=5)
    blk.train()
    x, coords = _canonical_tensor(geo, c, prec, seed=6)
    g = torch.randn((geo.n_out, c), device=DEV, generator=torch.Generator(device=DEV).manual_seed(8))
    before = _bn_states(blk)
    G.set_conv_precision(prec)
    try:
        xx = x.clone().requires_grad_(True)
        st = G.SparseConvTensor(xx, coords, geo.rb.in_shape, 2).canonical(assume_canonical=True)
        out = blk.conv1(st)
        out = out.replace_feature(blk.bn1(out.features))
        out = out.replace_feature(blk.relu(out.features))
        h = out.features
        out = blk.conv2(out)
        out = out.replace_feature(blk.bn2(out.features))
        out = out.replace_feature(out.features + st.features)
        out = out.replace_feature(blk.relu(out.features))
        out.features.backward(g)
    finally:
        G.set_conv_precision("fp32")
    l1, l2 = _ref_block(blk, before, x, geo, True, h.detach(), out.features.detach() > 0, prec)
    r1, r2 = _block_backward(l1, l2, g, c, prec)
    _compare_block(blk, xx, out.features.detach(), h.detach(), l1, l2, r1, r2, True, prec, f"unfused L2 {prec}")


# ---------------------------------------------------------------------------------------------- D. empty batches
def _empty_geo(cin, strided):
    ops = _ops()
    shape = [41, 200, 200]
    index = ops.OccupancyIndex(2, shape, torch.device(DEV, 0), "layers_empty")
    index.insert(torch.zeros((0, 4), dtype=torch.int32, device=DEV))
    index.build(0, known_n=0)
    if strided:
        rb, _ = ops.rulebook_sparse(index, [3, 3, 3], [2, 2, 2], [1, 1, 1], ("layers_empty", 1))
        return rb
    return ops.rulebook_subm(index, [3, 3, 3])


def _assert_empty_step(bns, params, nbt):
    for bn, (rm, rv) in bns:
        assert torch.equal(bn.running_mean, rm) and torch.equal(bn.running_var, rv)
        assert int(bn.num_batches_tracked) == nbt
    for name, p in params:
        assert p.grad is not None and not bool(p.grad.any()), name


@pytest.mark.parametrize("prec", PRECISIONS)
@pytest.mark.parametrize("strided", [False, True])
def test_conv_bn_act_empty_batch(strided, prec):
    """ops.conv_bn_act on zero rows: empty output, zero parameter gradients, running statistics unchanged,
    num_batches_tracked + 1 -- what torch.nn.BatchNorm1d does on an empty batch."""
    ops = _ops()
    print("data_ptr of an empty CUDA tensor:", torch.empty((0, 16), device=DEV).data_ptr())
    cin, cout = 16, 32
    rb = _empty_geo(cin, strided)
    bn = make_bn(cout, 0.5, 3)
    bn.train()
    stats = (bn.running_mean.clone(), bn.running_var.clone())
    x = torch.zeros((0, cin), device=DEV, requires_grad=True)
    w = torch.randn((cout, 3, 3, 3, cin), device=DEV, requires_grad=True)
    b = torch.randn((cout,), device=DEV, requires_grad=True)
    a, _ = ops.conv_bn_act(x, w, b, rb, _prec(prec), bn, None, True, None, prec == "bf16")
    assert a.shape == (0, cout)
    a.sum().backward()
    assert x.grad.shape == (0, cin)
    _assert_empty_step([(bn, stats)], [("w", w), ("b", b), ("gamma", bn.weight), ("beta", bn.bias)], 1)


@pytest.mark.parametrize("prec", PRECISIONS)
def test_res_block_empty_batch(prec):
    from toda_b200.spconv_compat import pytorch as G
    blk = _block(16, prec, seed=1)
    blk.train()
    stats = [(bn, (bn.running_mean.clone(), bn.running_var.clone())) for bn in (blk.bn1, blk.bn2)]
    x = torch.zeros((0, 16), device=DEV, requires_grad=True)
    G.set_conv_precision(prec)
    try:
        out = blk(G.SparseConvTensor(x, torch.zeros((0, 4), dtype=torch.int32, device=DEV), [41, 200, 200], 2))
        assert out.features.shape == (0, 16)
        out.features.sum().backward()
    finally:
        G.set_conv_precision("fp32")
    assert x.grad.shape == (0, 16)
    _assert_empty_step(stats, list(blk.named_parameters()), 1)


def test_sparse_sequential_empty_batch_counts_batchnorm():
    """SparseSequential(conv, BatchNorm1d, ReLU) as pcdet's post_act_block builds it: spconv skips the feature modules on
    an empty tensor; the BatchNorm still counts the batch, as torch does."""
    from toda_b200.spconv_compat import pytorch as G
    seq = G.SparseSequential(G.SubMConv3d(16, 16, 3, padding=1, bias=False, indice_key="e"), torch.nn.BatchNorm1d(16),
                             torch.nn.ReLU()).to(DEV).train()
    bn = seq[1]
    stats = (bn.running_mean.clone(), bn.running_var.clone())
    x = torch.zeros((0, 16), device=DEV, requires_grad=True)
    out = seq(G.SparseConvTensor(x, torch.zeros((0, 4), dtype=torch.int32, device=DEV), [41, 200, 200], 2))
    assert out.features.shape == (0, 16)
    assert torch.equal(bn.running_mean, stats[0]) and torch.equal(bn.running_var, stats[1])
    assert int(bn.num_batches_tracked) == 1


@pytest.mark.parametrize("prec", PRECISIONS)
def test_backbone_train_step_empty_batch(prec):
    """VoxelResBackBone8x forward, HeightCompression and backward on an all-empty batch of 2: an all-zero BEV map, an empty
    input gradient, zero parameter gradients, running statistics unchanged and every BatchNorm's batch counted."""
    import toda_b200.pcdet_plugin as P
    from toda_b200 import synth
    from toda_b200.spconv_compat import pytorch as G
    cfg = synth.CONFIGS["nus_0075"]
    grid = synth.grid_size_xyz(cfg["pc_range"], cfg["voxel_size"])
    torch.manual_seed(666)
    net = P.VoxelResBackBone8x(PU.Cfg(), 5, grid).to(DEV).train()
    hc = P.HeightCompression(PU.Cfg(NUM_BEV_FEATURES=256))
    bns = [(m, (m.running_mean.clone(), m.running_var.clone())) for m in net.modules() if isinstance(m, torch.nn.BatchNorm1d)]
    vf = torch.zeros((0, 5), device=DEV, requires_grad=True)
    G.set_conv_precision(prec)
    try:
        bd = hc(net({"voxel_features": vf, "voxel_coords": torch.zeros((0, 4), device=DEV), "batch_size": 2}))
        sf = bd["spatial_features"]
        assert sf.shape == (2, 256, int(grid[1]) // 8, int(grid[0]) // 8)
        assert not bool(sf.any())
        (sf * torch.randn(sf.shape, device=DEV)).sum().backward()
    finally:
        G.set_conv_precision("fp32")
    assert vf.grad.shape == (0, 5)
    _assert_empty_step(bns, list(net.named_parameters()), 1)
