"""Counts behind the live-item weight gradient (conv_tc_wgrad_kernel, csrc/conv_tc.cu), numpy only, no GPU.

The tensor-core wgrad splits the output rows of a convolution over the CTAs of one wave (wgrad_plan) and walks items = (row chunk, pass) pairs, a pass being a group of 128/Cin kernel offsets and a chunk 128 rows
(Cout <= 64) or 64 rows (Cout = 128).  An item is live when one of its offsets has a neighbour in the chunk's 128-row tile
(the rulebook's tile mask word).  For every wgrad shape of VoxelResBackBone8x on the bench's synthetic frames (4
nuScenes-shaped frames, rows in canonical (batch, z, y, x) order) this prints:
  * the fraction of items that are live;
  * items per CTA under even row splits (equal row counts): every item (what a walk of all items costs), and live items
    only (max / mean);
  * live items per CTA with the splits the kernel uses: each group's rows cut into ranges of whole row chunks holding
    equal shares of its live items (max / mean).
These are counts, not times: the slowest CTA of the single wave sets a launch's time, so max per CTA bounds the gain.

    python scripts/wgrad_live_items.py"""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from toda_b200 import synth  # noqa: E402

NUM_SMS = 148
FRAMES = 4


def level1_coords():
    """(batch, z, y, x) of the occupied voxels of the bench's frames, canonical order, and the grid (z, y, x)."""
    cfg = synth.CONFIGS["nus_0075"]
    frames, _ = synth.make_batch("nus_0075", FRAMES)
    r, vs = np.array(cfg["pc_range"], np.float32), np.array(cfg["voxel_size"], np.float32)
    grid = np.round((r[3:] - r[:3]) / vs).astype(np.int64)
    shape = np.array([grid[2] + 1, grid[1], grid[0]])
    out = []
    for b, pts in enumerate(frames):
        c = np.floor((np.asarray(pts)[:, 0:3] - r[:3]) / vs).astype(np.int64)
        c = c[((c >= 0) & (c < grid)).all(1)]
        zyx = np.unique(np.stack([c[:, 2], c[:, 1], c[:, 0]], 1), axis=0)
        out.append(np.concatenate([np.full((len(zyx), 1), b), zyx], 1))
    return np.concatenate(out), shape


def keys(c, shape):
    return ((c[:, 0] * shape[0] + c[:, 1]) * shape[1] + c[:, 2]) * shape[2] + c[:, 3]


def table(cin_coords, in_shape, out_coords, k, s, p):
    """Output-stationary neighbour table [kvol][n_out]: input row at out*s - p + offset, or -1."""
    kin = keys(cin_coords, in_shape)
    order = np.argsort(kin)
    sk = kin[order]
    rows = []
    for dz in range(k[0]):
        for dy in range(k[1]):
            for dx in range(k[2]):
                q = out_coords[:, 1:] * np.array(s) - np.array(p) + np.array([dz, dy, dx])
                inside = ((q >= 0) & (q < in_shape)).all(1)
                kk = keys(np.concatenate([out_coords[:, :1], q], 1), in_shape)
                idx = np.clip(np.searchsorted(sk, kk), 0, len(sk) - 1)
                hit = inside & (sk[idx] == kk)
                rows.append(np.where(hit, order[idx], -1))
    return np.stack(rows)


def downsample(coords, shape, k, s, p):
    out_shape = (shape + 2 * np.array(p) - np.array(k)) // np.array(s) + 1
    outs = []
    for dz in range(k[0]):
        for dy in range(k[1]):
            for dx in range(k[2]):
                o = coords[:, 1:] + np.array(p) - np.array([dz, dy, dx])
                ok = (o % np.array(s) == 0).all(1)
                o = o // np.array(s)
                ok &= ((o >= 0) & (o < out_shape)).all(1)
                outs.append(np.concatenate([coords[ok, :1], o[ok]], 1))
    u = np.unique(np.concatenate(outs), axis=0)      # lexicographic (batch, z, y, x): canonical order
    return u, out_shape


def tile_masks(nbr):
    kvol, n = nbr.shape
    t = (n + 127) // 128
    has = np.concatenate([nbr >= 0, np.zeros((kvol, t * 128 - n), bool)], 1).reshape(kvol, t, 128).any(2)
    return (has.astype(np.int64) << np.arange(kvol)[:, None]).sum(0)


def wgrad_plan(n_out, kvol, cin, cout):
    npad = 64 if cout <= 64 else 128
    rows = 128 if npad == 64 else 64
    offs = 128 // cin
    total = (kvol + offs - 1) // offs
    ppc = min(total, 512 // npad)
    groups = (total + ppc - 1) // ppc
    splits = max(1, min(max(1, NUM_SMS // groups), (n_out + 4 * rows - 1) // (4 * rows)))
    rps = max(rows, ((n_out + splits - 1) // splits + rows - 1) // rows * rows)
    return rows, offs, total, ppc, groups, splits, rps


def analyse(name, nbr, cin, cout):
    kvol, n = nbr.shape
    cin = max(cin, 16)
    rows, offs, total, ppc, groups, splits, rps = wgrad_plan(n, kvol, cin, cout)
    m = tile_masks(nbr)
    # live[c, q]: pass q has a neighbour in chunk c (its enclosing 128-row tile's word)
    nch = (n + rows - 1) // rows
    word = m[(np.arange(nch) * rows) >> 7]
    live = np.stack([((word >> (q * offs)) & ((1 << offs) - 1)) != 0 for q in range(total)], 1)
    even_all, even_live, bal_live = [], [], []
    for gi in range(groups):
        lg = live[:, gi * ppc:(gi + 1) * ppc]
        npass = lg.shape[1]
        for sp in range(splits):
            c0, c1 = sp * rps // rows, min(nch, (sp + 1) * rps // rows)
            even_all.append(max(0, c1 - c0) * npass)
            even_live.append(int(lg[c0:c1].sum()))
        # balanced as the kernel does it (wgrad_split_chunks): whole chunks, split s starting at the first chunk whose
        # preceding chunks hold floor(s*T/splits) of the group's T live items
        pre = np.concatenate([[0], np.cumsum(lg.sum(1))])
        t_live = int(pre[-1])
        bounds = [0] + [int(np.searchsorted(pre[:-1], sp * t_live // splits, side="left")) for sp in range(1, splits)] + [nch]
        bal_live += [int(pre[b1] - pre[b0]) for b0, b1 in zip(bounds[:-1], bounds[1:])]
    frac = live.sum() / max(1, live.size)
    print("| %-9s | %3d -> %3d | %6d | %2d x %3d | %5.1f %% | %4d | %4d / %6.1f | %4d / %6.1f |" % (
        name, cin, cout, n, groups, splits, 100 * frac, max(even_all), max(even_live), np.mean(even_live), max(bal_live),
        np.mean(bal_live)))


def main():
    c, s = level1_coords()
    print("Live (row chunk, pass) items of conv_tc_wgrad_kernel, %d synthetic nus_0075 frames (bench.py's first batch)\n" % FRAMES)
    print("| shape     | Cin -> Cout | rows   | grid     | live    | all items max/CTA | live, even splits max / mean "
          "| live, balanced splits max / mean |")
    print("|---|---|---|---|---|---|---|---|")
    # conv_input (4 -> 16, padded to 16 channels) and the SubM convs of level 1 share one table
    sub = table(c, s, c, (3, 3, 3), (1, 1, 1), (1, 1, 1))
    analyse("L1 subm", sub, 16, 16)
    levels = [((3, 3, 3), (2, 2, 2), (1, 1, 1), 16, 32), ((3, 3, 3), (2, 2, 2), (1, 1, 1), 32, 64),
              ((3, 3, 3), (2, 2, 2), (0, 1, 1), 64, 128)]
    for li, (k, st, p, ci, co) in enumerate(levels):
        o, os_ = downsample(c, s, k, st, p)
        analyse("down%d%d" % (li + 1, li + 2), table(c, s, o, k, st, p), ci, co)
        c, s = o, os_
        analyse("L%d subm" % (li + 2), table(c, s, c, (3, 3, 3), (1, 1, 1), (1, 1, 1)), co, co)
    o, os_ = downsample(c, s, (3, 1, 1), (2, 1, 1), (0, 0, 0))
    analyse("conv_out", table(c, s, o, (3, 1, 1), (2, 1, 1), (0, 0, 0)), 128, 128)


if __name__ == "__main__":
    main()
