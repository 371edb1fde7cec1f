"""Problem assembly just before the hot path (host side, numpy-vectorised).

Mirrors the contract of the reference's raster/network assembly so that the
Laplacian handed to the CUDA solver is the same matrix the reference would build:
  construct_node_map   src/raster/pairwise.jl:271-314
  construct_graph      src/raster/pairwise.jl:316-367
  laplacian            src/core.jl:608-634
  connected_components Graphs.connected_components (src/raster/pairwise.jl:214)
The synthetic-raster generator of the benchmark (SURVEY.md §8d) also lives here.
"""
from __future__ import annotations

import numpy as np
import scipy.sparse as sp
from scipy.sparse import csgraph


def construct_node_map(gmap, polymap=None):
    """Column-major numbering (1-based; 0 = no node) of cells with conductance > 0;
    every cell of a short-circuit polygon (NODATA ones too) takes the node of the
    polygon's first valid cell; labels are then compacted in order."""
    g = np.asarray(gmap)
    vf = (g > 0).reshape(-1, order="F")
    lab = np.zeros(vf.size, dtype=np.int64)
    lab[vf] = np.arange(1, int(vf.sum()) + 1)
    if polymap is not None and np.size(polymap):
        pf = np.asarray(polymap).reshape(-1, order="F").astype(np.int64)
        cand = np.nonzero((pf != 0) & vf)[0]                 # valid polygon cells, column-major
        if cand.size:
            pid, where = np.unique(pf[cand], return_index=True)   # first valid cell of each polygon
            rep = lab[cand[where]]
            pos = np.clip(np.searchsorted(pid, pf), 0, len(pid) - 1)
            hit = (pf != 0) & (pid[pos] == pf)
            lab[hit] = rep[pos[hit]]
        nz = lab != 0
        _, inv = np.unique(lab[nz], return_inverse=True)
        lab[nz] = inv + 1
    return lab.reshape(g.shape, order="F")


def create_new_polymap(gmap, polymap, points_rc, point_map):
    """Merge focal points into the short-circuit polygon map (one-to-all / all-to-one,
    src/raster/pairwise.jl:374-403): a focal id becomes a polygon of its own unless it
    already sits on one; focal *regions* overlapping a polygon take it over."""
    rr, cc, ids = points_rc
    if polymap is None or np.size(polymap) == 0:
        return np.array(point_map, dtype=np.int64)
    newpoly = np.array(polymap, dtype=np.int64)
    occupied = np.flatnonzero(np.asarray(point_map).reshape(-1, order="F"))
    cells = np.column_stack(np.unravel_index(occupied, point_map.shape, order="F"))
    if len(ids) == len(np.unique(ids)):
        k = int(np.max(polymap))
        for a, b in cells:
            if polymap[a, b] == 0:
                newpoly[a, b] = point_map[a, b] + k
        return newpoly
    k = max(int(np.max(polymap)), int(np.max(point_map)))
    for a, b in cells:
        v1, v2 = int(point_map[a, b]), int(newpoly[a, b])
        if v2 == 0:
            newpoly[a, b] = k + v1
        elif v1 != v2:
            newpoly[newpoly == v2] = v1
    return newpoly


def create_pair_polymap(gmap, polymap, points_rc, pt1, pt2):
    """Polygon map of one pair of focal REGIONS (pairwise with repeated focal ids,
    src/raster/pairwise.jl:405-442): without a polygon map every cell of pt1 / pt2 becomes a polygon
    named after its id; with one, a region of several cells that touches no polygon becomes a new
    polygon, and one that touches polygons merges all of them into a new polygon."""
    rr, cc, ids = (np.asarray(a) for a in points_rc)
    if polymap is None or np.size(polymap) == 0:
        newpoly = np.zeros(np.shape(gmap), dtype=np.int64)
        for p in (pt1, pt2):
            sel = ids == p
            newpoly[rr[sel] - 1, cc[sel] - 1] = p
        return newpoly
    polymap = np.asarray(polymap, dtype=np.int64)
    newpoly = polymap.copy()
    k = int(polymap.max())
    for p in (pt1, pt2):
        idx = np.nonzero(ids == p)[0]
        if len(idx) == 1:
            continue
        under = polymap[rr[idx] - 1, cc[idx] - 1]
        if np.all(under == 0):
            newpoly[rr[idx] - 1, cc[idx] - 1] = k + 1
            k += 1
            continue
        touched = under[under != 0]
        if len(touched) == 1:
            # the reference reads an undefined variable (`overlap`) on this branch and stops there
            raise ValueError(f"focal region {p} overlaps a short-circuit polygon in exactly one cell: "
                             "the reference cannot build its polygon map (UndefVarError)")
        newpoly[np.isin(polymap, touched)] = k + 1
        k += 1
    return newpoly


def construct_graph(gmap, nodemap, avg_res, four_neighbors):
    """Symmetric adjacency of conductances: E, S, SE, NE neighbours, duplicates
    (parallel cell adjacencies of merged nodes) summed."""
    g = np.asarray(gmap, dtype=np.float64)
    nm = np.asarray(nodemap)
    s2 = np.sqrt(2.0)
    if avg_res:
        f1 = lambda x, y: 1.0 / ((1.0 / x + 1.0 / y) / 2.0)
        f2 = lambda x, y: 1.0 / (s2 * (1.0 / x + 1.0 / y) / 2.0)
    else:
        f1 = lambda x, y: (x + y) / 2.0
        f2 = lambda x, y: (x + y) / (2.0 * s2)
    nr, nc = g.shape
    shifts = [((slice(None), slice(0, nc - 1)), (slice(None), slice(1, nc)), f1),
              ((slice(0, nr - 1), slice(None)), (slice(1, nr), slice(None)), f1)]
    if not four_neighbors:
        shifts += [((slice(0, nr - 1), slice(0, nc - 1)), (slice(1, nr), slice(1, nc)), f2),
                   ((slice(1, nr), slice(0, nc - 1)), (slice(0, nr - 1), slice(1, nc)), f2)]
    I, J, V = [], [], []
    with np.errstate(divide="ignore", invalid="ignore"):
        for a, b, f in shifts:
            na, nb = nm[a], nm[b]
            ok = (na != 0) & (nb != 0)
            I.append(na[ok] - 1)
            J.append(nb[ok] - 1)
            V.append(f(g[a], g[b])[ok])
    I, J, V = np.concatenate(I), np.concatenate(J), np.concatenate(V)
    m = int(nm.max())
    a = sp.coo_matrix((np.concatenate([V, V]), (np.concatenate([I, J]), np.concatenate([J, I]))),
                      shape=(m, m))
    return a.tocsr()


def laplacian(adj):
    """Off-diagonals -> -g_ij; diagonal -> sum_j g_ij (any stored diagonal dropped)."""
    a = sp.csr_matrix(adj, dtype=np.float64)
    a = a - sp.diags(a.diagonal())
    deg = np.asarray(a.sum(axis=1)).ravel()
    L = (sp.diags(deg) - a).tocsr()
    L.sort_indices()
    return L


def connected_components(G):
    """Components (1-based node ids, ascending), ordered by their smallest node."""
    A = sp.csr_matrix(G).copy()
    A.data = (A.data != 0).astype(np.int8)
    A.eliminate_zeros()
    ncomp, lab = csgraph.connected_components(A, directed=False)
    order = np.argsort(lab, kind="stable")
    counts = np.bincount(lab, minlength=ncomp)
    comps = np.split(order + 1, np.cumsum(counts)[:-1])
    comps.sort(key=lambda c: c[0])
    return comps


# ---------------------------------------------------------------------------
# synthetic benchmark problems (SURVEY.md §8d)
# ---------------------------------------------------------------------------
def synthetic_raster_laplacian(nrows, ncols, seed=42, four_neighbors=False, avg_res=False,
                               dtype=np.float64):
    """R ~ U[1,10] resistances -> g = 1/R; 8-neighbour average-conductance stencil;
    column-major node numbering.  Built directly in CSR (no COO pass) so the
    4000 x 4000 case (1.44e8 nnz) assembles in seconds and ~3 GB."""
    rng = np.random.default_rng(seed)
    g = 1.0 / rng.uniform(1.0, 10.0, size=(nrows, ncols))
    return stencil_laplacian_from_conductance(g, four_neighbors, avg_res, dtype), g


def stencil_laplacian_from_conductance(g, four_neighbors=False, avg_res=False, dtype=np.float64):
    """Laplacian of a full raster (every cell a node) straight into CSR."""
    g = np.asarray(g, dtype=np.float64)
    nr, nc = g.shape
    n = nr * nc
    s2 = np.sqrt(2.0)
    if avg_res:
        f1 = lambda x, y: 1.0 / ((1.0 / x + 1.0 / y) / 2.0)
        f2 = lambda x, y: 1.0 / (s2 * (1.0 / x + 1.0 / y) / 2.0)
    else:
        f1 = lambda x, y: (x + y) / 2.0
        f2 = lambda x, y: (x + y) / (2.0 * s2)
    # neighbour offsets (di, dj) in ascending node-id order for column-major numbering
    offs = [(-1, -1), (0, -1), (1, -1), (-1, 0), (1, 0), (-1, 1), (0, 1), (1, 1)]
    if four_neighbors:
        offs = [(0, -1), (-1, 0), (1, 0), (0, 1)]
    ii, jj = np.meshgrid(np.arange(nr), np.arange(nc), indexing="ij")
    ncolslots = len(offs) + 1
    vals = np.zeros((nr, nc, ncolslots))
    cols = np.full((nr, nc, ncolslots), -1, dtype=np.int64)
    diag_slot = len(offs) // 2
    deg = np.zeros((nr, nc))
    for k, (di, dj) in enumerate(offs):
        slot = k if k < diag_slot else k + 1
        ok = (ii + di >= 0) & (ii + di < nr) & (jj + dj >= 0) & (jj + dj < nc)
        src = g[ok]
        dst = g[(ii + di)[ok], (jj + dj)[ok]]
        w = f2(src, dst) if (di != 0 and dj != 0) else f1(src, dst)
        vals[..., slot][ok] = -w
        cols[..., slot][ok] = ((jj + dj) * nr + (ii + di))[ok]
        deg[ok] += w
    vals[..., diag_slot] = deg
    cols[..., diag_slot] = jj * nr + ii
    # to column-major row order
    vals = vals.transpose(1, 0, 2).reshape(n, ncolslots)
    cols = cols.transpose(1, 0, 2).reshape(n, ncolslots)
    keep = cols >= 0
    rowptr = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(keep.sum(axis=1), out=rowptr[1:])
    L = sp.csr_matrix((vals[keep].astype(dtype), cols[keep].astype(np.int32), rowptr.astype(np.int32 if rowptr[-1] < 2**31 else np.int64)),
                      shape=(n, n))
    return L


def power_law_laplacian(n, m=5, seed=11, dtype=np.float64):
    """Synthetic network-mode graph of SURVEY.md §8d / BASELINE config C5: preferential
    attachment (Barabasi-Albert style, m edges per new node, grown in batches that sample
    the degree-proportional endpoint list as of the batch start), conductances U[0.1, 1].
    Returns the CSR Laplacian of the (connected) graph.  The reference would get the same
    matrix from a 3-column network file through `laplacian!` (src/core.jl:608-624)."""
    rng = np.random.default_rng(seed)
    m0 = m + 1
    src = [np.repeat(np.arange(1, m0), np.arange(1, m0))]
    dst = [np.concatenate([np.arange(i) for i in range(1, m0)])]
    ends = np.concatenate([src[0], dst[0]])
    v0 = m0
    while v0 < n:
        nb = int(min(n - v0, max(1, v0 // 16)))
        v = np.repeat(np.arange(v0, v0 + nb), m)
        t = ends[rng.integers(0, len(ends), size=nb * m)]
        key = np.unique(v.astype(np.int64) * n + t)          # drop repeated targets of a node
        v, t = key // n, key % n
        src.append(v); dst.append(t)
        ends = np.concatenate([ends, v, t])
        v0 += nb
    s_, d_ = np.concatenate(src), np.concatenate(dst)
    w = rng.uniform(0.1, 1.0, len(s_))
    A = sp.coo_matrix((np.r_[w, w], (np.r_[s_, d_], np.r_[d_, s_])), shape=(n, n)).tocsr()
    L = (sp.diags(np.asarray(A.sum(axis=1)).ravel()) - A).tocsr().astype(dtype)
    L.sort_indices()
    return L


def focal_nodes(n, count, seed=7):
    """`count` distinct node ids (0-based) -- rng(7) as in SURVEY.md §8d."""
    rng = np.random.default_rng(seed)
    return np.sort(rng.choice(n, size=count, replace=False))


def all_pairs(nodes, limit=None):
    src, dst = [], []
    for a in range(len(nodes)):
        for b in range(a + 1, len(nodes)):
            src.append(nodes[a]); dst.append(nodes[b])
    src, dst = np.array(src, dtype=np.int64), np.array(dst, dtype=np.int64)
    if limit is not None:
        src, dst = src[:limit], dst[:limit]
    return src, dst
