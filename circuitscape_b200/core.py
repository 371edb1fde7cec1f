"""Drivers of the hot path on the CUDA solver -- the host-side mirror of
src/core.jl (pairwise) and src/raster/advanced.jl:151-333 (advanced).

Public names follow the reference:
    get_solver(cfg)                         src/core.jl:74-94
    single_ground_all_pairs(prob, flags, cfg)  src/core.jl:70-72  -> solve(...)
    advanced_kernel(prob, flags, cfg)       src/raster/advanced.jl:151-271
    multiple_solver(cfg, solver, a, s, g, f)   src/raster/advanced.jl:274-305
`solve(prob, ::CUDASolver)` is the batched direct-style driver (src/core.jl:312-515)
re-thought for a device-resident solver: the pair list of a component is handed to
ONE `cs_b200_solve_pairs` call; voltages, node currents and the cumulative/max
accumulation stay on the GPU and only resistances (plus whatever per-pair maps the
flags ask for) come back.
"""
from __future__ import annotations

import contextlib
from dataclasses import dataclass, field

import numpy as np
import scipy.sparse as sp

from . import solver as S

NODATA = -9999.0
RESISTANCE_INVALID = -777.0   # src/consts.jl:45


# ---------------------------------------------------------------------------
# config / selection  (src/config.jl:68-73, src/consts.jl:12-15, src/core.jl:74-94)
# ---------------------------------------------------------------------------
def _parse_solver(s):
    """Unknown names fall back to cg+amg in the reference; here the only product
    solver is the CUDA one, so anything outside the CUDA table is refused loudly."""
    if s in S.CUDAB200:
        return "st_cuda"
    raise ValueError(f"solver = {s!r} is not served by circuitscape_b200 "
                     f"(use one of {S.CUDAB200}; cg+amg/cholmod stay in Circuitscape.jl)")


def get_solver(cfg):
    _parse_solver(cfg.get("solver", "cuda"))
    return S.CUDASolver(
        bs=int(cfg.get("cholmod_batch_size", "1000")),
        precision=cfg.get("precision", "double"),
        device=int(cfg.get("gpu_device", "0")),
        rtol=float(cfg.get("gpu_rtol", "1e-6")),
        precond=cfg.get("gpu_preconditioner", "amg"),
    )


def _flag(cfg, key, default="false"):
    return cfg.get(key, default) in ("True", "true", "1")   # src/config.jl:55-57


@dataclass
class OutputFlags:
    """src/out.jl:1-10."""
    write_volt_maps: bool = False
    write_cur_maps: bool = False
    write_cum_cur_map_only: bool = False
    write_max_cur_maps: bool = False
    set_null_currents_to_nodata: bool = False
    set_null_voltages_to_nodata: bool = False
    compress_grids: bool = False
    log_transform_maps: bool = False

    @classmethod
    def from_cfg(cls, cfg):
        return cls(**{k: _flag(cfg, k) for k in cls.__dataclass_fields__})


@dataclass
class Flags:
    """RasterFlags / NetworkFlags (src/raster/pairwise.jl:1-12, src/network/pairwise.jl:84-92)."""
    is_raster: bool = True
    is_advanced: bool = False
    outputflags: OutputFlags = field(default_factory=OutputFlags)

    @classmethod
    def from_cfg(cls, cfg):
        return cls(is_raster=cfg.get("data_type", "raster") in ("raster", "Raster"),
                   is_advanced=cfg.get("scenario", "pairwise") in ("advanced", "Advanced"),
                   outputflags=OutputFlags.from_cfg(cfg))


@dataclass
class GraphProblem:
    """src/core.jl:10-22 (hbmeta dropped: file metadata is not on the path)."""
    G: sp.csr_matrix
    cc: list                      # list of 1-based node-id arrays
    points: np.ndarray            # graph node per focal point (1-based, 0 = none)
    user_points: np.ndarray       # user ids
    exclude_pairs: set = field(default_factory=set)
    nodemap: np.ndarray | None = None
    polymap: np.ndarray | None = None
    cellmap: np.ndarray | None = None
    solver: S.CUDASolver = field(default_factory=S.CUDASolver)
    coords: tuple | None = None   # network mode: (i, j) 1-based edge list (Cumulative.coords)


@dataclass
class PairwiseOutput:
    resistances: np.ndarray
    voltmaps: dict = field(default_factory=dict)
    curmaps: dict = field(default_factory=dict)
    branch: dict = field(default_factory=dict)
    cum_curmap: np.ndarray | None = None
    max_curmap: np.ndarray | None = None
    cum_node: np.ndarray | None = None
    cum_branch: np.ndarray | None = None
    num_solves: int = 0
    iterations: int = 0
    stats: list = field(default_factory=list)


# ---------------------------------------------------------------------------
# pair enumeration  (src/core.jl:386-424, 537-603)
# ---------------------------------------------------------------------------
def component_pairs(points, user_points, exclude, comp, shortcut):
    """For one component: unique focal nodes `csub` (in focal-point order), the
    node pairs to solve with their focal-index fan-out, and the index pairs that
    share a node (R = 0, smash_repeats!)."""
    points = np.asarray(points)
    member = np.isin(points, comp) & (points != 0)
    idx_by_node = {}
    for k in np.nonzero(member)[0]:
        idx_by_node.setdefault(int(points[k]), []).append(int(k))
    csub = list(idx_by_node)
    zero, solves = [], []
    for pi, s in enumerate(csub[: (1 if shortcut else len(csub))]):
        si = idx_by_node[s]
        zero += [(si[a], si[b]) for a in range(len(si)) for b in range(a + 1, len(si))]
        for d in csub[pi + 1:]:
            fan = [(ci, cj) for ci in si for cj in idx_by_node[d]
                   if (int(user_points[ci]), int(user_points[cj])) not in exclude]
            if fan:
                solves.append((s, d, fan))
    return csub, solves, zero


def construct_local_node_map(nodemap, comp, polymap):
    """src/utils.jl:10-30: cell -> row of the component's matrix (1-based, 0 = none)."""
    from .graph import construct_node_map
    inside = np.isin(nodemap, comp)
    local = np.where(inside, nodemap, 0)
    if np.array_equal(local, nodemap):
        return local
    if polymap is None or np.size(polymap) == 0:
        flat = local.reshape(-1, order="F")
        nz = flat != 0
        flat = flat.copy()
        flat[nz] = np.arange(1, int(nz.sum()) + 1)
        return flat.reshape(local.shape, order="F")
    return construct_node_map(local, np.where(inside, polymap, 0))


def _scatter(values, local_nodemap):
    out = np.zeros(local_nodemap.shape, dtype=np.float64)
    nz = local_nodemap != 0
    out[nz] = values[local_nodemap[nz] - 1]
    return out


def _process_grid(cmap, cellmap, log_transform, set_null_to_nodata):
    """src/out.jl:305-319."""
    if log_transform:
        pos = cmap > 0
        cmap = np.where(pos, np.log10(np.where(pos, cmap, 1.0)), NODATA)
    if set_null_to_nodata:
        cmap = np.where(cellmap == 0, NODATA, cmap)
    return cmap


# ---------------------------------------------------------------------------
# pairwise driver
# ---------------------------------------------------------------------------
def single_ground_all_pairs(prob: GraphProblem, flags: Flags, cfg=None, log=True, sink=None) -> PairwiseOutput:
    """src/core.jl:70-72."""
    return solve(prob, prob.solver, flags, cfg, log, sink=sink)


def _component_rows(nodemap, comp, polymap, n):
    """cell -> 1-based row of a whole-graph factor with n rows: the node whose value the component's
    local node map puts in the cell (row l of the component's submatrix is node comp[l]; with polygons
    the local numbering can differ from the submatrix's, and the maps follow the local numbering).
    Without polygons that is the cell's own node wherever it lies in the component."""
    if polymap is None or np.size(polymap) == 0:
        member = np.zeros(n + 1, dtype=bool)
        member[comp] = True
        return np.where(member[nodemap], nodemap, 0)
    lm = construct_local_node_map(nodemap, comp, polymap)
    return np.where(lm != 0, comp[np.maximum(lm, 1) - 1], 0)


def solve(prob: GraphProblem, solver: S.CUDASolver, flags: Flags, cfg=None, log=True, sink=None,
          factor=None) -> PairwiseOutput:
    """`sink`: optional writer the per-pair results are handed to as each batch finishes -- the
    reference writes every map inside `postprocess` and drops it (src/core.jl:655-683); without a
    sink they are kept in the returned object (tests, small jobs).  A sink has the methods
    `voltmap(key, grid)`, `curmap(key, grid)` (raster) and `network(key, comp, volt, cur, branch)`.

    `factor`: one resident factor whose row r is node r + 1 of the whole graph, e.g. a whole-raster
    handle (B200Factor.from_raster_polygons; block-diagonal over the components).  Every component's
    pairs are solved on it instead of on a factor of the component's submatrix, and the cumulative /
    max vectors are read back once for the job.  Raster mode only; `prob.G` is not used and
    `prob.cc` only needs the components that hold a focal node.  The caller keeps ownership."""
    shared = factor is not None
    if shared and not flags.is_raster:
        raise ValueError("solve(factor=...) serves raster problems only")
    o = flags.outputflags
    P = len(prob.points)
    R = -np.ones((P, P))
    want_maps = o.write_volt_maps or o.write_cur_maps or o.write_cum_cur_map_only or o.write_max_cur_maps
    shortcut = flags.is_raster and not want_maps and not prob.exclude_pairs      # src/core.jl:356-364
    voltmatrix = np.zeros((P, P))
    shortcut_res = -np.ones((P, P))
    out = PairwiseOutput(resistances=None)
    raster = flags.is_raster
    if raster:
        out.cum_curmap = np.zeros(prob.cellmap.shape)
        out.max_curmap = np.full(prob.cellmap.shape, NODATA) if o.write_max_cur_maps else None
    else:
        out.cum_node = np.zeros(prob.G.shape[0])
        out.cum_branch = np.zeros(len(prob.coords[0]))
        branch_pos = _BranchIndex(prob.coords)
    G = None if shared else sp.csr_matrix(prob.G)
    points = np.asarray(prob.points)
    ids = np.asarray(prob.user_points)
    if shared:
        factor.reset_currents()
        local_of = np.arange(-1, factor.n, dtype=np.int64)      # node id -> row of the shared factor
        rows_of_cells = np.asarray(prob.nodemap)                 # cell -> row + 1 read for the cumulative maps
        has_polygons = prob.polymap is not None and np.size(prob.polymap) > 0
        npost_total = 0.0

    for comp in prob.cc:
        comp = np.asarray(comp)
        csub, solves, zero = component_pairs(points, ids, prob.exclude_pairs, comp, shortcut)
        if not csub:
            continue
        for a, b in zero:
            R[a, b] = R[b, a] = 0.0
        if not solves:
            if shortcut:      # duplicates on the anchor only: the reference still runs the update (core.jl:504-506)
                anchor = int(np.nonzero(points == csub[0])[0][0])
                _update_shortcut_resistances(anchor, voltmatrix, shortcut_res, R, points, comp)
            continue
        rows = comp - 1
        if not shared:
            matrix = G[rows][:, rows].tocsr()
            local_of = np.zeros(G.shape[0] + 1, dtype=np.int64)
            local_of[comp] = np.arange(len(comp))
        src = np.array([local_of[s] for s, _, _ in solves])
        dst = np.array([local_of[d] for _, d, _ in solves])
        weight = np.array([len(f) for _, _, f in solves], dtype=np.float64)
        need_curr = not shortcut                       # postprocess always builds the current map
        per_pair_volt = o.write_volt_maps or (not raster and not shortcut)   # network branch currents need v
        per_pair_curr = need_curr and ((o.write_cur_maps and not o.write_cum_cur_map_only) or not raster)
        local_nodemap = None
        if raster and not shortcut and not shared:
            local_nodemap = construct_local_node_map(prob.nodemap, comp, prob.polymap)
        elif raster and not shortcut and (o.write_volt_maps or per_pair_curr or has_polygons):
            local_nodemap = _component_rows(prob.nodemap, comp, prob.polymap, factor.n)
        # only raster maps are log-transformed (src/out.jl:96 process_grid!); the network branch of
        # write_cur_maps accumulates raw node currents (src/out.jl:48-88)
        with (contextlib.nullcontext(factor) if shared else
              S.construct_cholesky_factor(matrix, solver, log_transform=bool(o.log_transform_maps and raster))) as factor:
            bs = max(1, int(solver.bs))
            if shortcut:
                inside = np.nonzero(np.isin(points, comp) & (points != 0))[0]
                focal_rows = np.unique(local_of[points[inside]])
                focal_col = {int(r): i for i, r in enumerate(focal_rows)}

            def batches():
                if getattr(solver, "superpose", False) and not shortcut and len(solves) > 1:
                    # one solve per focal NODE of the component, every pair by superposition
                    # (the Shortcut algebra of src/core.jl:685-739 applied to the voltages)
                    nodes, inv = np.unique(np.concatenate([src, dst]), return_inverse=True)
                    yield slice(0, len(solves)), factor.solve_pairs_superposed(
                        nodes, inv[:len(src)], inv[len(src):], weight, want_volt=per_pair_volt,
                        want_curr=per_pair_curr, accumulate=need_curr)
                    return
                for st in range(0, len(solves), bs):                            # src/core.jl:448-452
                    sl = slice(st, min(st + bs, len(solves)))
                    if shortcut:
                        # only the voltages at the focal nodes are used (update_voltmatrix!,
                        # src/core.jl:685-703): probe rows instead of n x k voltages over PCIe
                        res = factor.solve_sources([([s_, d_], [-1.0, 1.0]) for s_, d_ in zip(src[sl], dst[sl])],
                                                   ref=src[sl], probe=focal_rows)
                        res["R"] = np.array([res["probe_volt"][c, focal_col[d_]] for c, d_ in enumerate(dst[sl])])
                        yield sl, res
                        continue
                    yield sl, factor.solve_pairs(src[sl], dst[sl], weight[sl], want_volt=per_pair_volt,
                                                 want_curr=per_pair_curr, accumulate=need_curr)

            for sl, res in batches():
                out.stats.append(factor.stats())
                out.num_solves += len(res["R"])
                out.iterations += int(res["iters"].sum())
                for col, (s, d, fan) in enumerate(solves[sl]):
                    r = float(res["R"][col])
                    v = res["volt"][:, col].astype(np.float64) if res.get("volt") is not None else None
                    cur = res["curr"][:, col].astype(np.float64) if res.get("curr") is not None else None
                    br = _branch_currents(matrix, v, comp) if not raster and not shortcut else None
                    for ci, cj in fan:
                        R[ci, cj] = R[cj, ci] = r
                        key = (int(ids[ci]), int(ids[cj]))
                        if shortcut:                                             # src/core.jl:685-703
                            pv = res["probe_volt"][col]
                            for i in inside[inside >= 1]:
                                voltmatrix[i, cj] = 1.0 - float(pv[focal_col[int(local_of[points[i]])]]) / r
                            continue
                        if raster:
                            if o.write_volt_maps:
                                vm = _process_grid(_scatter(v, local_nodemap), prob.cellmap,
                                                   False, o.set_null_voltages_to_nodata)
                                if sink is not None:
                                    sink.voltmap(key, vm)
                                else:
                                    out.voltmaps[key] = vm
                            if per_pair_curr:
                                cm = _process_grid(_scatter(cur, local_nodemap), prob.cellmap,
                                                   o.log_transform_maps, o.set_null_currents_to_nodata)
                                if sink is not None:
                                    sink.curmap(key, cm)
                                else:
                                    out.curmaps[key] = cm
                        else:
                            # every id combination is post-processed on its own (src/core.jl:235-249):
                            # its branch currents go into the cumulative vector once each
                            branch_pos.add(out.cum_branch, br)
                            if sink is not None:
                                sink.network(key, comp, v if o.write_volt_maps else None, cur, br)
                            else:
                                if o.write_volt_maps:
                                    out.voltmaps[key] = (comp, v)
                                out.curmaps[key] = (comp, cur)
                                out.branch[key] = br
            if need_curr and shared:
                npost_total += float(weight.sum())
                if has_polygons:
                    rows_of_cells = np.where(local_nodemap != 0, local_nodemap, rows_of_cells)
            elif need_curr:
                cum, mx = factor.read_currents(want_max=True)
                if raster:
                    npost = float(weight.sum())
                    cmap = _scatter(cum.astype(np.float64), local_nodemap)
                    if o.log_transform_maps:
                        # cells outside the component hold 0 -> log-transformed to NODATA per pair
                        cmap = np.where(local_nodemap == 0, NODATA * npost, cmap)
                    if o.set_null_currents_to_nodata:
                        cmap = np.where(prob.cellmap == 0, NODATA * npost, cmap)
                    out.cum_curmap += cmap
                    if out.max_curmap is not None:
                        mmap = _scatter(mx.astype(np.float64), local_nodemap)
                        off = local_nodemap == 0
                        mmap = np.where(off, NODATA if o.log_transform_maps else 0.0, mmap)
                        if o.set_null_currents_to_nodata:
                            mmap = np.where(prob.cellmap == 0, NODATA, mmap)
                        out.max_curmap = np.maximum(out.max_curmap, mmap)
                else:
                    out.cum_node[rows] += cum
        if shortcut:
            anchor = int(np.nonzero(points == csub[0])[0][0])
            _update_shortcut_resistances(anchor, voltmatrix, shortcut_res, R, points, comp)
    if shared and npost_total > 0:
        _add_whole_raster_currents(out, factor, rows_of_cells, npost_total, prob.cellmap, o)
    if shortcut:
        R = shortcut_res
    np.fill_diagonal(R, 0.0)
    full = np.zeros((P + 1, P + 1))
    full[0, 1:] = ids
    full[1:, 0] = ids
    full[1:, 1:] = R
    out.resistances = full                                                      # src/core.jl:294-299
    if raster:
        out.cum_curmap = np.where(out.cum_curmap < NODATA, NODATA, out.cum_curmap)   # src/utils.jl:114-120
        if out.max_curmap is not None:
            out.max_curmap = np.where(out.max_curmap < NODATA, NODATA, out.max_curmap)
    return out


def _add_whole_raster_currents(out, factor, rows_of_cells, npost, cellmap, o):
    """The cumulative / max maps of a job solved on one whole-raster factor, from ONE read of its
    vectors.  Equal to the per-component sums of `solve` on per-component factors: a node outside a
    pair's component carries zero current (the 1e-8 relative zeroing removes the coupling noise of
    the coarse pseudo-inverse), which the log transform accumulates as NODATA once per post-processed
    pair -- what the per-component path adds for cells outside each component; cells without a node
    get NODATA times the job's count directly.  `rows_of_cells`: cell -> row + 1 (0 = no node)."""
    cum, mx = factor.read_currents(want_max=True)
    off = rows_of_cells == 0
    cmap = _scatter(cum.astype(np.float64), rows_of_cells)
    if o.log_transform_maps:
        cmap = np.where(off, NODATA * npost, cmap)
    if o.set_null_currents_to_nodata:
        cmap = np.where(cellmap == 0, NODATA * npost, cmap)
    out.cum_curmap += cmap
    if out.max_curmap is not None:
        mmap = np.where(off, NODATA if o.log_transform_maps else 0.0, _scatter(mx.astype(np.float64), rows_of_cells))
        if o.set_null_currents_to_nodata:
            mmap = np.where(cellmap == 0, NODATA, mmap)
        out.max_curmap = np.maximum(out.max_curmap, mmap)


def _focal_components(factor, points):
    """Components (1-based node ids, ascending) of a whole-graph factor that hold a focal node, in order
    of their smallest node, from the device labels (cs_b200_components)."""
    labels, _ = factor.components()
    pts = np.asarray(points, dtype=np.int64)
    pts = pts[pts != 0]
    return [np.flatnonzero(labels == c) + 1 for c in np.unique(labels[pts - 1])]


def raster_pairwise(cellmap, points_rc, flags: Flags, polymap=None, exclude_pairs=frozenset(), solver=None,
                    four_neighbors=False, avg_res=False, sink=None) -> PairwiseOutput:
    """Raster pairwise job from the conductance raster (src/raster/pairwise.jl:14-135), assembled,
    labelled and solved on the device.

    cellmap: conductances after masking (cells <= 0 are not nodes); points_rc: (rows, cols, ids)
    1-based, after include / exclude filtering; exclude_pairs: id pairs not to solve.  The output is
    that of `single_ground_all_pairs` on the host-built problem (resistances with the id header,
    per-pair maps or `sink`, cumulative / max maps, num_solves).

    Unique focal ids: ONE whole-raster factor (node map, Laplacian and components built on the
    device) serves every component's pairs.  Repeated ids (focal regions): one device assembly per
    pair on that pair's polygon map, as the reference rebuilds its graph per pair."""
    from . import graph
    solver = solver if solver is not None else S.CUDASolver()
    rr, cc_, ids = (np.asarray(a) for a in points_rc)
    log_t = bool(flags.outputflags.log_transform_maps)

    def run(poly, nodes, user_points, exclude):
        f, nodemap = S.B200Factor.from_raster_polygons(cellmap, poly, solver, four_neighbors=four_neighbors,
                                                       avg_res=avg_res, log_transform=log_t)
        with f:
            prob = GraphProblem(None, _focal_components(f, nodes(nodemap)), nodes(nodemap), user_points,
                                set(exclude), nodemap, poly, cellmap, solver)
            return solve(prob, solver, flags, sink=sink, factor=f)

    if len(ids) == len(np.unique(ids)):
        return run(polymap, lambda nm: nm[rr - 1, cc_ - 1], ids, exclude_pairs)

    pts = list(dict.fromkeys(int(p) for p in ids))
    first = {p: int(np.nonzero(ids == p)[0][0]) for p in pts}
    n = len(pts)
    R = -np.ones((n, n))
    out = None
    for i in range(n):
        for j in range(i + 1, n):
            p1, p2 = pts[i], pts[j]
            if (p1, p2) in exclude_pairs or (p2, p1) in exclude_pairs:
                continue
            x, y = first[p1], first[p2]
            r = run(graph.create_pair_polymap(cellmap, polymap, (rr, cc_, ids), p1, p2),
                    lambda nm: np.array([nm[rr[x] - 1, cc_[x] - 1], nm[rr[y] - 1, cc_[y] - 1]]),
                    np.array([p1, p2]), ())
            R[i, j] = R[j, i] = r.resistances[1, 2]
            if out is None:
                out = r
                continue
            out.voltmaps.update(r.voltmaps)
            out.curmaps.update(r.curmaps)
            out.cum_curmap = out.cum_curmap + r.cum_curmap
            if out.max_curmap is not None:
                out.max_curmap = np.maximum(out.max_curmap, r.max_curmap)
            out.num_solves += r.num_solves
            out.iterations += r.iterations
            out.stats += r.stats
    if out is None:                                       # every pair excluded
        out = PairwiseOutput(resistances=None, cum_curmap=np.zeros(np.shape(cellmap)),
                             max_curmap=np.full(np.shape(cellmap), NODATA)
                             if flags.outputflags.write_max_cur_maps else None)
    np.fill_diagonal(R, 0.0)
    full = np.zeros((n + 1, n + 1))
    full[0, 1:] = pts
    full[1:, 0] = pts
    full[1:, 1:] = R
    out.resistances = full
    return out


def _branch_currents(matrix, v, comp):
    """Network mode branch currents |G_ij| |v_i - v_j| over the stored upper triangle
    with the 1e-8 relative zeroing (src/out.jl:154-158, 250-290); host side, network
    graphs only.  Rows come in the order `_convert_to_3col` walks the CSC branch matrix
    (column-major: sorted by column, then row), so written files match the reference's."""
    coo = sp.triu(sp.csr_matrix(matrix), k=1).tocoo()
    order = np.lexsort((coo.row, coo.col))
    row, col, data = coo.row[order], coo.col[order], coo.data[order]
    b = np.abs(data) * (v[row] - v[col])
    if len(b):
        mx = b.max()
        with np.errstate(divide="ignore", invalid="ignore"):
            b = np.where(np.abs(b / mx) < 1e-8, 0.0, b)
    return comp[row], comp[col], np.abs(b)


class _BranchIndex:
    """Position of every graph edge in `coords` (the cumulative branch vector's order,
    src/utils.jl:132-142) by a sorted key table instead of the reference's linear `findfirst`
    per branch (src/out.jl:65-84).  An edge that is not in `coords` raises, like the reference's
    `cbc[nothing]`."""

    def __init__(self, coords):
        a = np.asarray(coords[0], dtype=np.int64)
        b = np.asarray(coords[1], dtype=np.int64)
        self.base = int(max(a.max(initial=0), b.max(initial=0))) + 1
        key = a * self.base + b
        # findfirst semantics: the first occurrence of a repeated edge wins
        self.order = np.argsort(key, kind="stable")
        self.keys = key[self.order]

    def _find(self, a, b):
        key = a * self.base + b
        pos = np.searchsorted(self.keys, key, side="left")
        ok = (pos < len(self.keys))
        ok[ok] = self.keys[pos[ok]] == key[ok]
        return np.where(ok, self.order[np.minimum(pos, len(self.keys) - 1)], -1)

    def add(self, cum, branch):
        gr, gc, val = branch
        gr = np.asarray(gr, dtype=np.int64)
        gc = np.asarray(gc, dtype=np.int64)
        k = self._find(gr, gc)
        miss = k < 0
        if miss.any():
            k[miss] = self._find(gc[miss], gr[miss])
        if (k < 0).any():
            i = int(np.nonzero(k < 0)[0][0])
            raise KeyError(f"branch ({int(gr[i])}, {int(gc[i])}) is not an edge of the graph")
        np.add.at(cum, k, val)


def _update_shortcut_resistances(anchor, voltmatrix, shortcut, resistances, points, comp):
    """src/core.jl:706-739:  R_2x = 2 R_12 V_x2 + R_1x - R_12."""
    check = np.isin(points, comp) & (np.asarray(points) != 0)
    l = resistances.shape[0]
    for px in np.nonzero(check)[0]:
        R1x = resistances[anchor, px]
        if R1x == -1:
            continue
        shortcut[px, anchor] = shortcut[anchor, px] = R1x
        for p2 in range(px, l):
            if not check[p2]:
                continue
            R12 = resistances[anchor, p2]
            if R12 == -1:
                continue
            if R1x != RESISTANCE_INVALID:
                shortcut[anchor, p2] = shortcut[p2, anchor] = R12
                R2x = 2 * R12 * voltmatrix[px, p2] + R1x - R12
                if shortcut[p2, px] != RESISTANCE_INVALID:
                    shortcut[p2, px] = shortcut[px, p2] = R2x
            else:
                shortcut[px, :] = RESISTANCE_INVALID
                shortcut[:, px] = RESISTANCE_INVALID


def compute_3col(r):
    """src/out.jl:12-26."""
    fp = r[1:, 0]
    i, j = np.triu_indices(len(fp), k=1)
    return np.column_stack([fp[i], fp[j], r[j + 1, i + 1]])


# ---------------------------------------------------------------------------
# advanced mode  (src/raster/advanced.jl:151-333)
# ---------------------------------------------------------------------------
@dataclass
class AdvancedProblem:
    """src/raster/advanced.jl:1-15."""
    G: sp.csr_matrix
    cc: list
    sources: np.ndarray
    grounds: np.ndarray
    finitegrounds: np.ndarray       # [-9999.] sentinel when there are none
    nodemap: np.ndarray | None = None
    polymap: np.ndarray | None = None
    cellmap: np.ndarray | None = None
    solver: S.CUDASolver = field(default_factory=S.CUDASolver)


@dataclass
class AdvancedOutput:
    voltages: np.ndarray
    voltmap: np.ndarray | None = None
    curmap: np.ndarray | None = None
    node_currents: np.ndarray | None = None
    branch: tuple | None = None


def multiple_solver(cfg, solver, a, sources, grounds, finitegrounds, resident=None):
    """src/raster/advanced.jl:274-305: diag += finite grounds; rows/cols of Inf
    grounds deleted (0 V); `multiple_solve`; zeros re-inserted.

    resident = (cache dict, key): keep ONE device factor of the component's Laplacian `a` under `key`
    and move the grounds on the device (cs_b200_set_grounds: identity rows instead of deleted ones)
    -- for the one-to-all / all-to-one loops, where only the grounds change between iterations."""
    if resident is not None:
        cache, key = resident
        f = cache.get(key)
        if f is None:
            f = cache[key] = S.construct_cholesky_factor(sp.csr_matrix(a, dtype=np.float64), solver)
        mask = np.asarray(grounds) == np.inf
        f.set_grounds(None if finitegrounds[0] == NODATA else np.asarray(finitegrounds, dtype=np.float64),
                      mask if mask.any() else None)
        b = np.asarray(sources, dtype=np.float64).copy()
        b[mask] = 0.0
        v = np.asarray(S.solve_linear_system(f, a, b), dtype=np.float64).copy()   # residual gate inside (hook #2)
        v[mask] = 0.0
        return v
    a = sp.csr_matrix(a, dtype=np.float64)
    n = a.shape[0]
    if finitegrounds[0] != NODATA:
        a = (a + sp.diags(finitegrounds)).tocsr()
    keep = np.nonzero(~(grounds == np.inf))[0]
    asolve = a[keep][:, keep].tocsr()
    volt = S.multiple_solve(solver, asolve, np.asarray(sources, dtype=np.float64)[keep])
    v = np.zeros(n)
    v[keep] = volt
    return v


def node_currents_host(G, v, finitegrounds=None):
    """src/out.jl:178-207 on the host (advanced mode solves once per component; the
    pairwise path uses the device kernel instead)."""
    coo = sp.triu(sp.csr_matrix(G), k=1).tocoo()
    n = G.shape[0]
    d = np.abs(coo.data) * (v[coo.row] - v[coo.col])

    def one(b):
        if len(b):
            mx = b.max()
            with np.errstate(divide="ignore", invalid="ignore"):
                b = np.where(np.abs(b / mx) < 1e-8, 0.0, b)
        s = np.zeros(n)
        np.add.at(s, coo.col, np.maximum(b, 0.0))
        np.add.at(s, coo.row, np.maximum(-b, 0.0))
        return s

    p, q = one(d), one(-d)
    if finitegrounds is not None and finitegrounds[0] != NODATA:
        fg = finitegrounds * v
        p = p + np.where(fg < 0, -fg, 0.0)
        q = q + np.where(fg > 0, fg, 0.0)
    return np.where(p > q, p, q)


def advanced_kernel(prob: AdvancedProblem, flags: Flags, cfg=None) -> AdvancedOutput:
    G = sp.csr_matrix(prob.G)
    n = G.shape[0]
    raster = flags.is_raster
    voltages = np.zeros(n)
    outvolt = np.zeros(prob.nodemap.shape) if raster else None
    outcurr = np.zeros(prob.nodemap.shape) if raster else None
    for c in prob.cc:
        rows = np.asarray(c) - 1
        s_local, g_local = prob.sources[rows].copy(), prob.grounds[rows].copy()
        if s_local.sum() == 0 or g_local.sum() == 0:                          # :194-196
            continue
        f_local = prob.finitegrounds[rows] if prob.finitegrounds[0] != NODATA else prob.finitegrounds
        a_local = G[rows][:, rows].tocsr()
        voltages[rows] += multiple_solver(cfg, prob.solver, a_local, s_local, g_local, f_local)
        if raster:
            lm = construct_local_node_map(prob.nodemap, np.asarray(c), prob.polymap)
            outvolt += _scatter(voltages[rows], lm)
            outcurr += _scatter(node_currents_host(a_local, voltages[rows], f_local), lm)
    res = AdvancedOutput(voltages, outvolt, outcurr)
    if not raster:
        res.node_currents = node_currents_host(G, voltages, prob.finitegrounds)
        res.branch = _branch_currents(G, voltages, np.arange(1, n + 1))
    return res


def all_to_one_batched(factor, focal, rtol=None, shard=None, device_resident=False, accumulate=False):
    """All-to-one on a graph WITHOUT finite grounds, batched on one factor.

    Iteration c of the reference's all-to-one loop (src/raster/onetoall.jl:110-118,146-151)
    ties focal node f_c to ground (Dirichlet, row/column deleted in `multiple_solver`,
    src/raster/advanced.jl:286-300) and injects 1 A at every other focal node.  Current
    conservation makes that the singular-Laplacian system  L v = e_others - (P-1) e_fc
    followed by the shift v -= v[f_c] -- the pairwise trick of src/core.jl:224-232 with a
    multi-source right-hand side -- so every iteration shares ONE operator and the P
    solves are columns of one batch instead of P factorizations.  `factor` must hold the
    connected component's Laplacian; `shard=(rank, world)` keeps columns rank::world.

    device_resident=False: through hook #2 (`solve_linear_system`, n x k host batch);
        returns (voltages (n, P'), iters, relres, cols).
    device_resident=True: through cs_b200_solve_sources -- right-hand sides are scattered
        on the device, only the voltages at the focal nodes come back, node currents are
        accumulated into the handle's cumulative / max vectors when `accumulate`;
        returns (focal voltages (P', P), iters, relres, cols)."""
    focal = np.asarray(focal, dtype=np.int64)
    cols = np.arange(len(focal)) if shard is None else np.arange(shard[0], len(focal), shard[1])
    n = factor.n
    if device_resident:
        columns = []
        for c in cols:
            v = np.ones(len(focal))
            v[c] = -(len(focal) - 1.0)
            columns.append((focal, v))
        o = factor.solve_sources(columns, focal[cols], probe=focal, accumulate=accumulate, rtol=rtol)
        return o["probe_volt"], o["iters"], o["relres"], cols
    rhs = np.zeros((n, len(cols)), dtype=factor.io_dtype, order="F")
    for j, c in enumerate(cols):
        rhs[focal, j] = 1.0
        rhs[focal[c], j] = -(len(focal) - 1.0)
    x, iters, relres = factor.solve_rhs(rhs, rtol=rtol)
    x = np.asarray(x).reshape(n, len(cols))
    x -= x[focal[cols], np.arange(len(cols))][None, :]
    return x, iters, relres, cols


# ---------------------------------------------------------------------------
# one-to-all / all-to-one  (src/raster/onetoall.jl) -- callers of the advanced kernel
# ---------------------------------------------------------------------------
def compute_omniscape_current(conductance, source, ground, cs_cfg, solver=None):
    """src/utils.jl:145-257 -- Omniscape's moving-window solve: one advanced-mode solve per
    connected component of a conductance window, returning the node-current raster.

    conductance / source / ground: 2-D arrays of one shape (NODATA or 0 conductance = no
    node; ground values are conductances: the reference hard-wires grnd_file_is_res =
    false, policy :rmvsrc and the average-conductance rule there, utils.jl:190-193);
    cs_cfg: the INI dictionary (only `connect_four_neighbors_only` and the solver keys are
    read).  `solver` overrides `get_solver(cs_cfg)`; tests pass a CPU double here."""
    from . import graph
    cellmap = np.array(conductance, dtype=np.float64)
    cellmap[cellmap == NODATA] = 0.0
    nodemap = graph.construct_node_map(cellmap, None)
    four = _flag(cs_cfg, "connect_four_neighbors_only")
    G = graph.laplacian(graph.construct_graph(cellmap, nodemap, False, four))
    cc = graph.connected_components(G)
    s, g, f = sources_and_grounds_from_maps(np.asarray(source, dtype=np.float64),
                                            np.asarray(ground, dtype=np.float64), nodemap, G.shape[0], "rmvsrc")
    prob = AdvancedProblem(G, cc, s, g, f, nodemap, None, cellmap, solver if solver is not None else get_solver(cs_cfg))
    return advanced_kernel(prob, Flags(is_raster=True, is_advanced=True), cs_cfg).curmap


def resolve_conflicts(sources, grounds, policy):
    """src/raster/advanced.jl:119-149 (`rmvall` only zeroes the sources -- pinned upstream by
    test/internal.jl:130-135)."""
    sources = np.array(sources, dtype=np.float64)
    grounds = np.array(grounds, dtype=np.float64)
    finite = np.where(np.isfinite(grounds), grounds, 0.0)
    if not np.any(finite != 0):
        finite = np.array([NODATA])
    both = (sources != 0) & (grounds != 0)
    if policy in ("rmvsrc", "rmvall"):
        sources[both] = 0
    elif policy == "rmvgnd":
        grounds[both] = 0
    grounds[np.isinf(grounds) & (sources > 0)] = 0
    return sources, grounds, finite


def sources_and_grounds_from_maps(source_map, ground_map, nodemap, n, policy):
    """src/raster/advanced.jl:81-117 (raster branch): cell values accumulate on their node."""
    sources = np.zeros(n)
    grounds = np.zeros(n)
    for target, cmap in ((sources, source_map), (grounds, ground_map)):
        sel = (cmap != 0) & (nodemap != 0)
        np.add.at(target, nodemap[sel] - 1, cmap[sel])
    return resolve_conflicts(sources, grounds, policy)


@dataclass
class RasterData:
    """The fields of src/io.jl:34-43 the one-to-all driver reads."""
    cellmap: np.ndarray
    polymap: np.ndarray | None
    points_rc: tuple                 # (rows, cols, ids) 1-based, sorted by id
    strengths: np.ndarray | None = None       # (P, 2) id, strength
    included_pairs: object | None = None      # .mode, .point_ids, .mat


@dataclass
class OneToAllOutput:
    resistances: np.ndarray
    curmaps: dict = field(default_factory=dict)
    voltmaps: dict = field(default_factory=dict)
    cum_curmap: np.ndarray | None = None
    max_curmap: np.ndarray | None = None
    num_solves: int = 0


def _one_to_all_batched_raster(G, comps, nodemap, newpoly, point_map, unique_point_map, uniq, rr, cc_,
                               strengths, solver):
    """One-to-all without include/exclude lists: iteration p puts a current source on focal node p and
    ties every OTHER focal node to ground (src/raster/onetoall.jl:100-109).  With F the focal nodes of
    a component and N the rest, all iterations share B = L[N, N] (the Laplacian with every focal
    row/column deleted, SPD); block elimination of the one live focal node gives
        B w_p = -L[N, p] ,   v_p = s_p / (L[p, p] + L[p, N] w_p) ,   v_N = v_p w_p ,   v = 0 on the other focal nodes,
    so the iterations of a component are columns of ONE n_N x |F| batch on one factor (hook #2) instead
    of one factor + solve per iteration.  Returns {iteration: (voltage raster, current raster,
    source-cell voltage / strength)}; iterations it cannot serve take the per-iteration path."""
    n_nodes = G.shape[0]
    if strengths is not None and len(strengths) != len(uniq):
        return {}
    comp_of = np.zeros(n_nodes + 1, dtype=np.int64) - 1
    for ci, comp in enumerate(comps):
        comp_of[np.asarray(comp)] = ci
    plans = {}
    for i, n in enumerate(uniq):
        if point_map.sum() == n:
            continue
        strv = float(strengths[i, 1]) if strengths is not None else 1.0
        source_map = np.where(unique_point_map == n, strv, 0.0)
        ground_map = np.where((point_map != n) & (point_map > 0), np.inf, 0.0)
        s_, g_, f_ = sources_and_grounds_from_maps(source_map, ground_map, nodemap, n_nodes, "rmvgnd")
        check_node = nodemap[rr[i] - 1, cc_[i] - 1]
        snodes = np.nonzero(s_ != 0)[0]
        if len(snodes) != 1 or f_[0] != NODATA or check_node == 0 or not np.all(np.isinf(g_[g_ != 0])):
            continue
        ci = comp_of[check_node]
        if ci < 0 or comp_of[snodes[0] + 1] != ci:
            continue
        rows = np.asarray(comps[ci]) - 1
        if not np.any(np.isinf(g_[rows])):
            continue                                   # no ground in this component: nothing is solved
        plans.setdefault(ci, []).append((i, int(snodes[0]), float(s_[snodes[0]]),
                                         frozenset(np.nonzero(np.isinf(g_[rows]))[0].tolist())))
    served = {}
    for ci, items in plans.items():
        rows = np.asarray(comps[ci]) - 1
        local = np.zeros(n_nodes, dtype=np.int64) - 1
        local[rows] = np.arange(len(rows))
        a_local = G[rows][:, rows].tocsr()
        F = sorted({int(local[p]) for _, p, _, _ in items} | set().union(*[g for *_x, g in items]))
        # every served iteration must ground exactly F minus its own source node
        items = [it for it in items if it[3] == frozenset(F) - {int(local[it[1]])}]
        if not items or len(F) >= len(rows):
            continue
        Nidx = np.setdiff1d(np.arange(len(rows)), F)
        B = a_local[Nidx][:, Nidx].tocsr()
        cols = [int(local[p]) for _, p, _, _ in items]
        rhs = -a_local[Nidx][:, cols].toarray()
        if not np.any(rhs):
            continue
        live = np.nonzero(np.abs(rhs).sum(axis=0) > 0)[0]
        W = np.zeros_like(rhs)
        with S.construct_cholesky_factor(B, solver) as factor:
            W[:, live] = np.asarray(S.solve_linear_system(factor, B, np.asfortranarray(rhs[:, live]))).reshape(len(Nidx), -1)
        lm = construct_local_node_map(nodemap, np.asarray(comps[ci]), newpoly)
        for c, (i, p, sval, _) in enumerate(items):
            pl = cols[c]
            lpn = a_local[pl, Nidx].toarray().ravel()
            denom = a_local[pl, pl] + lpn @ W[:, c]
            v = np.zeros(len(rows))
            v[pl] = sval / denom
            v[Nidx] = v[pl] * W[:, c]
            cur = node_currents_host(a_local, v, None)
            # the reported value is read off the voltage RASTER at the source cell, through the local
            # node map, exactly as the per-iteration path does (advanced.jl:252-263) -- with a NODATA
            # cell inside a focal region the local numbering can differ from the matrix's
            volt = np.zeros(lm.shape)
            volt[lm != 0] = v[lm[lm != 0] - 1]
            smap = np.where(unique_point_map == uniq[i], sval, 0.0)
            val = (volt[smap != 0] / smap[smap != 0])[0]
            served[i] = (_scatter(v, lm), _scatter(cur, lm), val)
    return served


def _all_to_one_batched_raster(G, comps, nodemap, newpoly, point_map, unique_point_map, uniq, rr, cc_,
                                strengths, solver, o):
    """All-to-one without include/exclude lists: every iteration keeps the same node map and operator
    and differs only in which focal node is tied to ground, so the iterations of one connected
    component are columns of ONE sparse-RHS batch on the component's singular Laplacian
    (cs_b200_solve_sources; ground = reference row carrying minus the summed sources) instead of
    one factor + solve per iteration (src/raster/onetoall.jl:110-151 through
    src/raster/advanced.jl:274-305).  Returns {iteration index: (voltage raster, current raster)}
    for the iterations it could serve; the caller runs the rest through the per-iteration path."""
    n_nodes = G.shape[0]
    strength_map = None
    if strengths is not None:
        strength_map = np.zeros(point_map.shape)
        strength_map[rr - 1, cc_ - 1] = strengths[:, 1] if len(strengths) == len(rr) else 0.0
        if len(strengths) != len(rr):
            return {}
    plans = {}      # component index -> list of (iteration, ground node, source nodes, source values)
    comp_of = np.zeros(n_nodes + 1, dtype=np.int64) - 1
    for ci, comp in enumerate(comps):
        comp_of[np.asarray(comp)] = ci
    for i, n in enumerate(uniq):
        if point_map.sum() == n:
            continue
        if strength_map is not None:
            source_map = np.where(unique_point_map == n, 0.0, strength_map)
        else:
            source_map = np.where((unique_point_map != 0) & (point_map != n), 1.0, 0.0)
        ground_map = np.where(point_map == n, np.inf, 0.0)
        s_, g_, f_ = sources_and_grounds_from_maps(source_map, ground_map, nodemap, n_nodes, "rmvsrc")
        gnodes = np.nonzero(np.isinf(g_))[0]
        check_node = nodemap[rr[i] - 1, cc_[i] - 1]
        if len(gnodes) != 1 or f_[0] != NODATA or check_node == 0:
            continue                                   # several ground nodes: per-iteration path
        ci = comp_of[check_node]
        if ci < 0 or comp_of[gnodes[0] + 1] != ci:
            continue
        rows = np.asarray(comps[ci]) - 1
        local = np.zeros(n_nodes, dtype=np.int64) - 1
        local[rows] = np.arange(len(rows))
        src_nodes = np.nonzero(s_[rows] != 0)[0]
        if len(src_nodes) == 0:
            continue
        plans.setdefault(ci, []).append((i, int(local[gnodes[0]]), src_nodes, s_[rows][src_nodes]))
    served = {}
    for ci, items in plans.items():
        rows = np.asarray(comps[ci]) - 1
        a_local = G[rows][:, rows].tocsr()
        lm = construct_local_node_map(nodemap, np.asarray(comps[ci]), newpoly)
        columns, refs = [], []
        for _, gl, sn, sv in items:
            columns.append((np.concatenate([sn, [gl]]), np.concatenate([sv, [-sv.sum()]])))
            refs.append(gl)
        with S.construct_cholesky_factor(a_local, solver) as factor:
            r = factor.solve_sources(columns, refs, want_volt=True, want_curr=True)
        for c, (i, *_rest) in enumerate(items):
            served[i] = (_scatter(r["volt"][:, c].astype(np.float64), lm),
                         _scatter(r["curr"][:, c].astype(np.float64), lm))
    return served


def onetoall_kernel(data: RasterData, flags: Flags, cfg, solver=None, one_to_all=None,
                    four_neighbors=False, avg_res=False) -> OneToAllOutput:
    """src/raster/onetoall.jl:13-167.  One advanced-mode solve per focal id: one-to-all = unit
    (or variable-strength) source at the focal node, every other focal node a direct ground;
    all-to-one = the reverse.  Every solve goes through `multiple_solver` -> hook #3."""
    from . import graph
    solver = solver or get_solver(cfg)
    if one_to_all is None:
        one_to_all = cfg.get("scenario") in ("one-to-all", "one_to_all")
    o = flags.outputflags
    gmap, polymap = data.cellmap, data.polymap
    rr, cc_, ids = (np.asarray(a) for a in data.points_rc)
    strengths = None if data.strengths is None else np.array(data.strengths, dtype=np.float64)
    inc = data.included_pairs
    mode = 0 if (inc is not None and inc.mode == "include") else 1
    if inc is not None:
        keep = np.isin(ids, inc.point_ids)
        rr, cc_, ids = rr[keep], cc_[keep], ids[keep]
        if strengths is not None:
            strengths = strengths[np.isin(strengths[:, 0], inc.point_ids)]
    points_rc = (rr, cc_, ids)
    point_map = np.zeros(gmap.shape, dtype=np.int64)
    point_map[rr - 1, cc_ - 1] = ids
    uniq = list(dict.fromkeys(int(p) for p in ids))
    newpoly = graph.create_new_polymap(gmap, polymap, points_rc, point_map)
    nodemap = graph.construct_node_map(gmap, newpoly)
    adj = graph.construct_graph(gmap, nodemap, avg_res, four_neighbors)
    comps = graph.connected_components(adj)
    G = graph.laplacian(adj)
    first = {p: int(np.nonzero(ids == p)[0][0]) for p in uniq}
    unique_point_map = np.zeros(gmap.shape, dtype=np.int64)
    for p, k in first.items():
        unique_point_map[rr[k] - 1, cc_[k] - 1] = p
    out = OneToAllOutput(resistances=None)
    out.cum_curmap = np.zeros(gmap.shape)
    out.max_curmap = np.full(gmap.shape, NODATA) if o.write_max_cur_maps else None
    res = np.zeros(len(uniq))
    strength_map = np.zeros(gmap.shape) if strengths is not None else None
    batched = {}
    if (not one_to_all) and inc is None and getattr(solver, "batch_all_to_one", False):
        batched = _all_to_one_batched_raster(G, comps, nodemap, newpoly, point_map, unique_point_map, uniq,
                                             rr, cc_, strengths, solver, o)
    batched1 = {}
    if one_to_all and inc is None and getattr(solver, "batch_one_to_all", False):
        batched1 = _one_to_all_batched_raster(G, comps, nodemap, newpoly, point_map, unique_point_map, uniq,
                                              rr, cc_, strengths, solver)
    resident_factors = {}          # CUDASolver(resident_grounds=True): one device factor per component
    for i, n in enumerate(uniq):
        pm, nm, npoly = point_map.copy(), nodemap, newpoly
        if inc is not None:
            for j, other in enumerate(inc.point_ids):
                if i != j and inc.mat[i, j] == mode:
                    pm[pm == int(other)] = 0
            npoly = graph.create_new_polymap(gmap, polymap, points_rc, pm)
            nm = graph.construct_node_map(gmap, polymap)            # (sic) onetoall.jl:88
        if strengths is not None:
            st = strengths.copy()
            st[pm[rr - 1, cc_ - 1] == 0, 1] = 1
            strength_map[rr - 1, cc_ - 1] = st[:, 1]
        if pm.sum() == n:                                           # no other focal node left
            res[i] = -1
            continue
        if i in batched1:                                           # one-to-all column of the grounded batch
            outvolt, outcurr, val = batched1[i]
            out.num_solves += 1
            res[i] = -1 if np.isclose(val, 0) else val               # advanced.jl:252-263
            if o.write_volt_maps:
                out.voltmaps[n] = outvolt
            if o.write_cur_maps or o.write_cum_cur_map_only:
                out.curmaps[n] = outcurr
            out.cum_curmap += outcurr
            if out.max_curmap is not None:
                out.max_curmap = np.maximum(out.max_curmap, outcurr)
            continue
        if i in batched:                                            # solved as a column of the batch
            outvolt, outcurr = batched[i]
            out.num_solves += 1
            res[i] = 0
            if o.write_volt_maps:
                out.voltmaps[n] = outvolt
            if o.write_cur_maps or o.write_cum_cur_map_only:
                out.curmaps[n] = outcurr
            out.cum_curmap += outcurr
            if out.max_curmap is not None:
                out.max_curmap = np.maximum(out.max_curmap, outcurr)
            continue
        if one_to_all:
            strv = strengths[i, 1] if strengths is not None else 1.0
            source_map = np.where(unique_point_map == n, float(strv), 0.0)
            ground_map = np.where((pm != n) & (pm > 0), np.inf, 0.0)
            policy = "rmvgnd"
        else:
            if strengths is not None:
                source_map = np.where(unique_point_map == n, 0.0, strength_map)
            else:
                source_map = np.where((unique_point_map != 0) & (pm != n), 1.0, 0.0)
            ground_map = np.where(pm == n, np.inf, 0.0)
            policy = "rmvsrc"
        check_node = nm[rr[i] - 1, cc_[i] - 1]                      # (sic) row i of points_rc
        s_, g_, f_ = sources_and_grounds_from_maps(source_map, ground_map, nm, G.shape[0], policy)
        volt = np.zeros(gmap.shape)
        outvolt, outcurr, called = np.zeros(gmap.shape), np.zeros(gmap.shape), False
        for comp in comps:
            if check_node not in comp:                               # advanced.jl:186-188
                continue
            rows = np.asarray(comp) - 1
            sl, gl = s_[rows].copy(), g_[rows].copy()
            if sl.sum() == 0 or gl.sum() == 0:
                continue
            fl = f_[rows] if f_[0] != NODATA else f_
            a_local = G[rows][:, rows].tocsr()
            v = multiple_solver(cfg, solver, a_local, sl, gl, fl,
                                resident=(resident_factors, tuple(rows[:2]) + (len(rows),))
                                if getattr(solver, "resident_grounds", False) else None)
            out.num_solves += 1
            lm = construct_local_node_map(nm, np.asarray(comp), npoly)
            called = True
            outvolt += _scatter(v, lm)
            outcurr += _scatter(node_currents_host(a_local, v, fl), lm)
            volt[lm != 0] = v[lm[lm != 0] - 1]
        if not called:
            res[i] = -1                                              # advanced.jl:246-250
        elif one_to_all:
            val = volt[source_map != 0] / source_map[source_map != 0]
            res[i] = -1 if np.isclose(val[0], 0) else val[0]         # advanced.jl:252-263
        else:
            res[i] = 0
        if o.write_volt_maps:
            out.voltmaps[n] = outvolt
        if o.write_cur_maps or o.write_cum_cur_map_only:
            out.curmaps[n] = outcurr
        out.cum_curmap += outcurr
        if out.max_curmap is not None:
            out.max_curmap = np.maximum(out.max_curmap, outcurr)
    for f in resident_factors.values():
        f.close()
    out.resistances = np.column_stack([uniq, res])
    out.cum_curmap = np.where(out.cum_curmap < NODATA, NODATA, out.cum_curmap)
    return out
