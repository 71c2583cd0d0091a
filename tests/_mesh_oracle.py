"""numpy float32 restatement of the surface-extraction rules of include/b2nerf.h (b2n_mesh_*) / DESIGN.md §5f, written
from the rules, not from the kernel: marching tetrahedra over the 6 Kuhn tetrahedra of every cell of the lattice padded
with a sigma = 0 ring.  Also the mesh checks (2-manifold and orientation, Euler characteristic, volume) and a few analytic
fields shared by the CPU and GPU mesh tests."""
import itertools

import numpy as np
import torch

F32 = np.float32
# direction classes in vertex order, as (dx, dy, dz)
DIRS = [(1, 0, 0), (0, 1, 0), (0, 0, 1), (1, 1, 0), (1, 0, 1), (0, 1, 1), (1, 1, 1)]
# the permutations (a, b, c) of the axes in lexicographic order; tetrahedron = {0, e_a, e_a+e_b, e_a+e_b+e_c}
PERMS = list(itertools.permutations(range(3)))


def parity(seq):
    """0 for an even permutation, 1 for an odd one"""
    s = 0
    for i in range(len(seq)):
        for j in range(i + 1, len(seq)):
            s ^= int(seq[i] > seq[j])
    return s


def tet_corners(perm):
    """the 4 local vertices of the tetrahedron of ``perm`` as 0/1 offsets within the cell"""
    a, b, _ = perm
    v1 = [0, 0, 0]
    v1[a] = 1
    v2 = list(v1)
    v2[b] = 1
    return [(0, 0, 0), tuple(v1), tuple(v2), (1, 1, 1)]


def tet_triangles(case, odd):
    """triangles of one tetrahedron as triples of local edges (m, n), m < n.  ``case`` bit m = local vertex m inside;
    ``odd`` = the tetrahedron (v0, v1, v2, v3) is negatively oriented.  Winding: normal from inside to outside."""
    ins = [m for m in range(4) if case >> m & 1]
    out = [m for m in range(4) if not case >> m & 1]

    def e(a, b):
        return (min(a, b), max(a, b))
    if len(ins) == 1:                                   # around the inside corner, facing away from it
        i, (j, k, l) = ins[0], out
        if parity((i, j, k, l)):
            k, l = l, k
        tris = [(e(i, j), e(i, k), e(i, l))]
    elif len(ins) == 3:                                 # around the outside corner, facing towards it
        o, (a, b, c) = out[0], ins
        if parity((o, a, b, c)):
            b, c = c, b
        tris = [(e(o, a), e(o, c), e(o, b))]
    elif len(ins) == 2:                                 # quad (ik, il, jl, jk), diagonal ik - jl
        (i, j), (k, l) = ins, out
        if parity((i, j, k, l)):
            k, l = l, k
        tris = [(e(i, k), e(i, l), e(j, l)), (e(i, k), e(j, l), e(j, k))]
    else:
        tris = []
    if odd:
        tris = [(t[0], t[2], t[1]) for t in tris]
    return tris


def extended_axis(axis):
    """axis [R] (fp32) -> [R+2] with axis[0] - h and axis[R-1] + h, h = axis[1] - axis[0] in fp32"""
    axis = np.asarray(axis, dtype=F32)
    h = F32(axis[1] - axis[0])
    return np.concatenate([[F32(axis[0] - h)], axis, [F32(axis[-1] + h)]]).astype(F32)


def extract(sigma, tau, axis):
    """(verts [V,3] float32, faces [F,3] int32) of the rules; sigma [R,R,R], axis [R] = the lattice's 1-D axis"""
    sigma = np.asarray(sigma, dtype=F32)
    tau = F32(tau)
    R = sigma.shape[0]
    N = R + 2
    ext = extended_axis(axis)
    s = np.zeros((N + 1, N + 1, N + 1), F32)            # one more zero layer: p + d past the ring reads 0 (no crossing)
    s[1:R + 1, 1:R + 1, 1:R + 1] = sigma
    ins = s > tau
    P = np.stack(np.meshgrid(np.arange(N), np.arange(N), np.arange(N), indexing="ij"), -1)     # [N,N,N,3]
    cross = np.zeros((N, N, N, 7), bool)
    for d, (dx, dy, dz) in enumerate(DIRS):
        cross[..., d] = ins[:N, :N, :N] != ins[dx:N + dx, dy:N + dy, dz:N + dz]
    flat = cross.reshape(-1)
    vid = np.full(flat.shape, -1, np.int64)
    sel = np.nonzero(flat)[0]                           # ordered by point, then direction class
    vid[sel] = np.arange(len(sel))
    vid = vid.reshape(N, N, N, 7)
    pidx, d = np.divmod(sel, 7)
    p = np.stack(np.unravel_index(pidx, (N, N, N)), -1)
    q = p + np.array(DIRS)[d]
    ext_pad = np.concatenate([ext, [F32(0)]])           # index N is never a vertex end (no crossing there)
    sa = s[p[:, 0], p[:, 1], p[:, 2]]
    sb = s[q[:, 0], q[:, 1], q[:, 2]]
    t = (tau - sa) / (sb - sa)
    pa, pb = ext_pad[p], ext_pad[q]
    verts = (pa + t[:, None] * (pb - pa)).astype(F32)
    # faces: cells = lowest points with every coordinate <= R
    C = P[:N - 1, :N - 1, :N - 1].reshape(-1, 3)
    cell_lin = (C[:, 0] * N + C[:, 1]) * N + C[:, 2]
    rows = []                                           # (cell_lin, tet, slot, v0, v1, v2)
    dir_of = {dv: k for k, dv in enumerate(DIRS)}
    for ti, perm in enumerate(PERMS):
        lv = tet_corners(perm)
        odd = parity(perm)
        case = np.zeros(len(C), np.int64)
        for m in range(4):
            o = np.array(lv[m])
            c = C + o
            case |= ins[c[:, 0], c[:, 1], c[:, 2]].astype(np.int64) << m
        for cs in range(16):
            at = np.nonzero(case == cs)[0]
            if len(at) == 0:
                continue
            for slot, tri in enumerate(tet_triangles(cs, odd)):
                ids = []
                for (m, n) in tri:
                    o = np.array(lv[m])
                    dd = dir_of[tuple(np.array(lv[n]) - o)]
                    c = C[at] + o
                    ids.append(vid[c[:, 0], c[:, 1], c[:, 2], dd])
                rows.append(np.stack([cell_lin[at], np.full(len(at), ti), np.full(len(at), slot)] + ids, -1))
    if not rows:
        return verts.reshape(-1, 3), np.zeros((0, 3), np.int32)
    rows = np.concatenate(rows)
    rows = rows[np.lexsort((rows[:, 2], rows[:, 1], rows[:, 0]))]
    faces = rows[:, 3:]
    assert (faces >= 0).all()
    return verts, faces.astype(np.int32)


# ------------------------------------------------------------------ checks
def check_closed_manifold(verts, faces):
    """every undirected edge belongs to exactly two faces that traverse it in opposite directions; every vertex is
    used; returns (V, E, F).  Works on CPU or CUDA tensors / numpy arrays."""
    f = torch.as_tensor(faces).long()
    V = int(torch.as_tensor(verts).shape[0])
    F = int(f.shape[0])
    if F == 0:
        return V, 0, 0
    a = f.reshape(-1)
    b = f.roll(-1, dims=1).reshape(-1)
    assert bool((a != b).all()), "degenerate face (repeated vertex id)"
    key = torch.sort(a * V + b).values
    assert bool((key[1:] != key[:-1]).all()), "a directed edge is used by two faces"
    rev = torch.sort(b * V + a).values
    assert torch.equal(key, rev), "an edge is not traversed once in each direction"
    used = torch.zeros(V, dtype=torch.bool, device=f.device)
    used[a] = True
    assert bool(used.all()), "unused vertex"
    return V, key.numel() // 2, F


def euler(verts, faces):
    V, E, F = check_closed_manifold(verts, faces)
    return V - E + F


def signed_volume(verts, faces):
    v = torch.as_tensor(verts).double()
    f = torch.as_tensor(faces).long()
    a, b, c = v[f[:, 0]], v[f[:, 1]], v[f[:, 2]]
    return float((a * torch.linalg.cross(b, c, dim=1)).sum() / 6.0)


# ------------------------------------------------------------------ analytic fields (sigma = 1 + slope * signed distance)
TAU = 1.0


def grid_points(axis):
    ax = torch.as_tensor(axis, dtype=torch.float64)
    return torch.meshgrid(ax, ax, ax, indexing="ij")


def sdf(name, x, y, z):
    """signed distance (positive inside) of the analytic test shapes, float64"""
    def ball(cx, cy, cz, r):
        return r - torch.sqrt((x - cx) ** 2 + (y - cy) ** 2 + (z - cz) ** 2)
    if name == "ball":
        return ball(0.05, -0.03, 0.02, 0.6)
    if name == "torus":
        q = torch.sqrt(x ** 2 + y ** 2) - 0.55
        return 0.22 - torch.sqrt(q ** 2 + z ** 2)
    if name == "two_balls":
        return torch.maximum(ball(-0.45, 0.0, 0.0, 0.35), ball(0.45, 0.1, 0.0, 0.3))
    if name == "slab":                                  # |x| < 0.3, cut by the four box faces in y and z
        return 0.3 - x.abs() + 0.0 * y
    raise KeyError(name)


ANALYTIC_VOLUME = {"ball": 4 / 3 * np.pi * 0.6 ** 3, "torus": 2 * np.pi ** 2 * 0.55 * 0.22 ** 2,
                   "two_balls": 4 / 3 * np.pi * (0.35 ** 3 + 0.3 ** 3)}
ANALYTIC_AREA = {"ball": 4 * np.pi * 0.6 ** 2, "torus": 4 * np.pi ** 2 * 0.55 * 0.22,
                 "two_balls": 4 * np.pi * (0.35 ** 2 + 0.3 ** 2)}
EULER = {"ball": 2, "torus": 0, "two_balls": 4, "slab": 2}


def field(name, axis, seed=0):
    """sigma [R,R,R] float32 (torch, CPU) of a named test field on the lattice of ``axis``"""
    x, y, z = grid_points(axis)
    R = x.shape[0]
    if name == "empty":
        return torch.zeros(R, R, R)
    if name == "full":
        return torch.full((R, R, R), 2.0 * TAU)
    if name == "noise":                                  # i.i.d. around tau: every tetrahedron case occurs
        g = torch.Generator().manual_seed(seed)
        return (TAU + (torch.rand(R, R, R, generator=g) - 0.5)).float()
    return (TAU + 4.0 * sdf(name, x, y, z)).float()
