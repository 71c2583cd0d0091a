#!/usr/bin/env python
"""How much the 16 points of a warp share table entries and sectors in the spatially ordered hash-grid kernels, per level
(CPU only, about a minute).  DESIGN.md section 7b.

Sample set: the C2 bench's (synthetic.random_rays(2^18), 128 jittered samples per ray between 2 and 6, every sample inside
the box: dense occupancy), ordered by the Morton key of b2n_hash_order (cell on a 2^7 lattice over the box; inside a bucket
the points keep ray order), cut into the 16-point warps of the pair-lane kernels (lanes 2i / 2i+1: point i, x = 0 / 1
column).  Geometry: L = 16, base 16, per-level scale 1.5, T = 2^19, F = 2 (4 entries per 32-byte sector).  Counts are per
point over a random sample of warps:

  run-merged   table-gradient reductions of the run merging (ray order's rule, offset slots): a run of points in the same
               cell is merged 2^steps points at a time below res 128, every corner is reduced on its own above
  inst-entries distinct entries per instruction (4 instructions, one per (y, z) corner slot), summed: the reductions of
               the warp-level entry merge when the slots are by OFFSET (dy, dz)
  par-entries  the same with the slots by vertex PARITY ((cy + dy) & 1, (cz + dz) & 1): the entry merge of the ordered
               scatter (k_hash_bwd_table_pair)
  warp-entries distinct entries of the warp's 128 corner contributions: the floor of any merge
  sec-offset   distinct 32-byte sectors per gather instruction, summed, slots by offset (L1TEX line visits of the gather
               before the parity slots)
  sec-parity   the same with the parity slots (k_hash_fwd_pair on ordered input)
  warp-sectors distinct sectors of the whole warp

    python tools/hash_sharing.py [n_warps]
"""
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "project-nerf_b200")]
import torch  # noqa: E402

from b2n import synthetic  # noqa: E402
from b2n.ops import HashGeometry  # noqa: E402

BOUND, ORDER_BITS, MERGE_RES = 1.5, 7, 128


def sample_set(B=2 ** 18, N=128):
    ro, rd, _ = synthetic.random_rays(B, seed=0)
    u = torch.rand(B, N, generator=torch.Generator().manual_seed(1))
    z = 2.0 + (torch.arange(N).float() + u) * (4.0 / N)
    pts = (ro[:, None, :] + rd[:, None, :] * z[..., None]).reshape(-1, 3).numpy()
    pts = pts[np.all(np.abs(pts) <= BOUND, axis=1)]
    return np.clip((pts + BOUND) / np.float32(2 * BOUND), 0, 1).astype(np.float32)


def morton_order(x01, bits=ORDER_BITS):
    q = np.minimum((x01 * (1 << bits)).astype(np.uint64), (1 << bits) - 1)
    key = np.zeros(len(q), np.uint64)
    for b in range(bits):
        for d in range(3):
            key |= ((q[:, d] >> np.uint64(b)) & np.uint64(1)) << np.uint64(3 * b + d)
    return np.argsort(key, kind="stable")


def n_distinct(a):
    """distinct values along the last axis, summed over the rest"""
    s = np.sort(a.reshape(-1, a.shape[-1]), axis=1)
    return int(s.shape[0] + (np.diff(s, axis=1) != 0).sum())


def run_merged(cell, res):
    """reductions per warp of the run merging of k_hash_bwd_table_pair on offset slots (every point with a gradient)"""
    if res > MERGE_RES:
        return 8 * cell.size
    steps = 4 if res <= 54 else (3 if res <= 122 else 2)
    head = np.ones_like(cell, dtype=bool)
    head[:, 1:] = cell[:, 1:] != cell[:, :-1]
    run_start = np.maximum.accumulate(np.where(head, np.arange(16)[None, :], 0), axis=1)
    issuers = ((np.arange(16)[None, :] - run_start) % (1 << steps)) == 0
    return 8 * int(issuers.sum())


def main(n_warps=100_000):
    t0 = time.time()
    x01 = sample_set()
    perm = morton_order(x01)
    P = len(perm)
    rng = np.random.default_rng(0)
    ws = rng.choice(P // 16, n_warps, replace=False)
    xs = x01[perm[(ws[:, None] * 16 + np.arange(16)[None, :]).reshape(-1)]]
    geom = HashGeometry(16, 16, 1.5, 19, 2)
    n = n_warps * 16
    print(f"{P} points in the box ({time.time() - t0:.0f} s); {n_warps} random warps of 16 points; per point:")
    cols = ("run-merged", "inst-entries", "par-entries", "warp-entries", "sec-offset", "sec-parity", "warp-sectors")
    print(f"{'level':>5} {'res':>5} {'kind':>6} " + " ".join(f"{c:>12}" for c in cols))
    tot = np.zeros(len(cols))
    for l, (scale, res, size, offset, hashed) in enumerate(geom.levels):
        pos = xs * np.float32(scale) + np.float32(0.5)
        g = np.floor(pos).astype(np.uint64)
        cx, cy, cz = g[:, 0], g[:, 1], g[:, 2]
        # ent[w, slot k, lane]: lane = 2 point + x column; offset slots k = dy + 2 dz, parity slots k = vy & 1 + 2 (vz & 1)
        ent_off = np.empty((n_warps, 4, 32), np.uint64)
        ent_par = np.empty((n_warps, 4, 32), np.uint64)
        for dy in (0, 1):
            for dz in (0, 1):
                vy, vz = cy + np.uint64(dy), cz + np.uint64(dz)
                par = ((vy & np.uint64(1)) | ((vz & np.uint64(1)) << np.uint64(1))).reshape(n_warps, 16)
                for s in (0, 1):
                    vx = cx + np.uint64(s)
                    if hashed:
                        e = (vx ^ ((vy * np.uint64(2654435761)) & np.uint64(0xffffffff))
                             ^ ((vz * np.uint64(805459861)) & np.uint64(0xffffffff))) & np.uint64(size - 1)
                    else:
                        e = (vx + vy * np.uint64(res) + vz * np.uint64(res * res)) % np.uint64(size)
                    e = (e + np.uint64(offset)).reshape(n_warps, 16)
                    ent_off[:, dy + 2 * dz, s::2] = e
                    # every point has one corner of each parity: scatter by parity into the slot
                    for k in range(4):
                        m = par == k
                        ent_par[:, k, s::2] = np.where(m, e, ent_par[:, k, s::2])
        cell = (cx + cy * np.uint64(res) + cz * np.uint64(res * res)).reshape(n_warps, 16)
        row = np.array([run_merged(cell, res), n_distinct(ent_off), n_distinct(ent_par),
                        n_distinct(ent_off.reshape(n_warps, 128)), n_distinct(ent_off // np.uint64(4)),
                        n_distinct(ent_par // np.uint64(4)), n_distinct(ent_off.reshape(n_warps, 128) // np.uint64(4))],
                       dtype=np.float64) / n
        tot += row
        print(f"{l:5d} {res:5d} {'hashed' if hashed else 'dense':>6} " + " ".join(f"{v:12.2f}" for v in row), flush=True)
    print(f"{'all':>5} {'':>5} {'':>6} " + " ".join(f"{v:12.2f}" for v in tot))
    print(f"({time.time() - t0:.0f} s)")


if __name__ == "__main__":
    main(int(sys.argv[1]) if len(sys.argv) > 1 else 100_000)
