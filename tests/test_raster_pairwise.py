"""circuitscape_b200.raster_pairwise: pairwise raster jobs assembled, labelled (cs_b200_components) and
solved from the conductance raster on one whole-raster factor.

CPU: the labelling kernels of csrc/components.cuh restated in Python against scipy; the driver with a
whole-raster CPU double (host assembly, each pair solved on its own component) against the goldens and
against the host-built path of tests/cases.py; graph.create_pair_polymap against the oracle.
GPU: the device labels against graph.connected_components; the goldens on the device; a multi-component
raster against single_ground_all_pairs on the host-built problem."""
import numpy as np
import pytest
import scipy.sparse as sp

import circuitscape_b200 as cb
from circuitscape_b200 import graph
from circuitscape_b200 import solver as S
from oracle import circuitscape_oracle as co

from . import cases
from .fake_factor import FakeFactor

NODATA = -9999.0


# ---- the labelling algorithm, restated ----------------------------------------------------------------
def emulate_components(A, rng):
    """k_cc_init / k_cc_hook / k_cc_flatten / scan / k_cc_label of components.cuh with the 'threads'
    of the hooking pass run in a random order (the result must not depend on it)."""
    A = sp.csr_matrix(A)
    n = A.shape[0]
    rp, ci, va = A.indptr, A.indices, A.data
    parent = np.arange(n)
    for v in range(n):
        for j in range(rp[v], rp[v + 1]):
            if ci[j] < parent[v] and va[j] != 0:
                parent[v] = ci[j]

    def find_root(v):
        cur = parent[v]
        if cur == v:
            return v
        prev = v
        while cur > parent[cur]:
            nxt = parent[cur]
            parent[prev] = nxt
            prev, cur = cur, nxt
        return cur

    for v in rng.permutation(n):
        for j in range(rp[v], rp[v + 1]):
            u = ci[j]
            if u == v or va[j] == 0:
                continue
            a, b = find_root(v), find_root(u)
            while a != b:
                if a < b:
                    a, b = b, a
                if parent[a] == a:               # atomicCAS(parent + a, a, b)
                    parent[a] = b
                    break
                a = find_root(parent[a])
    assert np.all(parent <= np.arange(n))
    for v in range(n):
        r = parent[v]
        while parent[r] != r:
            r = parent[r]
        parent[v] = r
    flag = np.append((parent == np.arange(n)).astype(np.int64), 0)
    ordinal = np.cumsum(flag) - flag
    return ordinal[parent], int(ordinal[n])


def labels_of(comps, n):
    lab = np.empty(n, dtype=np.int32)
    for c, comp in enumerate(comps):
        lab[np.asarray(comp) - 1] = c
    return lab


def island_raster(rng, nr, nc, holes=0.3):
    """islands, isolated cells, and cells linked to others only through a diagonal"""
    g = rng.uniform(0.2, 3.0, (nr, nc))
    g[rng.random((nr, nc)) < holes] = 0.0
    g[:, nc // 2] = 0.0                                   # a NODATA column: at least two islands
    g[nr // 2, :] = 0.0                                   # NODATA, as the masked cellmap holds it
    if nr > 4 and nc > 4:
        g[0:3, 0:3] = 0.0
        g[0, 0] = g[1, 1] = 1.0                           # diagonal-only link: two components with four neighbours
    return g


def island_polygons(rng, g):
    """a polygon bridging the islands across the NODATA column and row"""
    nr, nc = g.shape
    poly = np.zeros(g.shape, dtype=np.int64)
    poly[nr // 2 - 1: nr // 2 + 2, nc // 2 - 1: nc // 2 + 2] = 3
    poly[rng.integers(0, nr, 4), rng.integers(0, nc, 4)] = 5
    return poly


@pytest.mark.parametrize("seed", range(8))
@pytest.mark.parametrize("four", [False, True])
@pytest.mark.parametrize("polygons", [False, True])
def test_labelling_restated_on_cpu(seed, four, polygons):
    rng = np.random.default_rng(seed)
    g = island_raster(rng, int(rng.integers(5, 14)), int(rng.integers(5, 14)))
    poly = island_polygons(rng, g) if polygons else None
    nodemap = graph.construct_node_map(g, poly)
    A = graph.laplacian(graph.construct_graph(g, nodemap, False, four))
    comps = graph.connected_components(A)
    want = labels_of(comps, A.shape[0])
    for order_seed in range(3):
        got, ncomp = emulate_components(A, np.random.default_rng(order_seed))
        assert ncomp == len(comps) and np.array_equal(got, want)


def test_labelling_restated_on_cpu_diagonal_only_link():
    g = np.zeros((4, 4))
    g[0, 0] = g[1, 1] = g[3, 3] = 1.0
    for four, expect in ((False, [0, 0, 1]), (True, [0, 1, 2])):
        nm = graph.construct_node_map(g, None)
        A = graph.laplacian(graph.construct_graph(g, nm, False, four))
        got, ncomp = emulate_components(A, np.random.default_rng(0))
        assert list(got) == expect and ncomp == max(expect) + 1


# ---- the driver on a CPU double of the whole-raster factor ----------------------------------------------
class RasterFactorDouble(FakeFactor):
    """CPU double of a whole-raster B200Factor: the host assembly (graph.py) stands in for the device's,
    graph.connected_components for cs_b200_components; each pair is solved on its own component (the
    whole-raster Laplacian is singular per component) and its voltages / currents are zero elsewhere,
    which is what the device's 1e-8 zeroing leaves there."""

    def __init__(self, conductance, polymap, solver, four_neighbors=False, avg_res=False, log_transform=False):
        g = np.where(np.asarray(conductance) > 0, conductance, 0.0)
        self.nodemap = graph.construct_node_map(g, polymap).astype(np.int32)
        L = graph.laplacian(graph.construct_graph(g, self.nodemap, avg_res, four_neighbors))
        super().__init__(L, solver, log_transform)
        self.comps = graph.connected_components(L)
        self.labels = labels_of(self.comps, self.n)

    def components(self):
        return self.labels.copy(), len(self.comps)

    def _rows(self, node):
        return np.asarray(self.comps[self.labels[node]]) - 1

    def solve_pairs(self, src, dst, weight=None, want_volt=False, want_curr=False, accumulate=False, **kw):
        src, dst = np.asarray(src), np.asarray(dst)
        k = len(src)
        w = np.ones(k) if weight is None else np.asarray(weight, dtype=float)
        V, curr = np.zeros((self.n, k)), np.zeros((self.n, k))
        for c in range(k):
            rows = self._rows(src[c])
            local = {int(r): i for i, r in enumerate(rows)}
            sub = self.A[rows][:, rows]
            V[rows, c] = co.solve_pairs_direct(sub, [local[int(src[c])]], [local[int(dst[c])]])[:, 0]
            curr[rows, c] = co.get_node_currents(sub, V[rows, c])
            if accumulate:
                val = np.where(curr[:, c] > 0, np.log10(np.where(curr[:, c] > 0, curr[:, c], 1.0)), NODATA) \
                    if self.log else curr[:, c]
                self.cum += w[c] * val
                self.mx = np.maximum(self.mx, val)
        R = V[dst, np.arange(k)] - V[src, np.arange(k)]
        return dict(R=R, volt=V if want_volt else None, curr=curr if want_curr else None,
                    iters=np.zeros(k, dtype=np.int64), relres=np.zeros(k))

    def solve_sources(self, columns, ref, probe=None, **kw):
        k = len(columns)
        V = np.zeros((self.n, k))
        for c, (r_, v_) in enumerate(columns):
            rows = self._rows(ref[c])
            local = np.full(self.n, -1)
            local[rows] = np.arange(len(rows))
            sub = FakeFactor(self.A[rows][:, rows], self.solver)
            one = sub.solve_sources([(local[np.asarray(r_, dtype=np.int64)], v_)], [local[ref[c]]],
                                    probe=np.arange(len(rows)))
            V[rows, c] = one["probe_volt"][0]
        pv = None if probe is None else V[np.asarray(probe)].T.copy()
        return dict(probe_volt=pv, volt=None, curr=None, iters=np.zeros(k, dtype=np.int64), relres=np.zeros(k))


@pytest.fixture
def cpu_device(monkeypatch):
    made = []

    def from_raster_polygons(conductance, polymap, solver, four_neighbors=False, avg_res=False, log_transform=False):
        f = RasterFactorDouble(conductance, polymap, solver, four_neighbors, avg_res, log_transform)
        made.append(f)
        return f, f.nodemap.copy()

    monkeypatch.setattr(S.B200Factor, "from_raster_polygons", staticmethod(from_raster_polygons))
    monkeypatch.setattr(S, "construct_cholesky_factor", lambda m, s, **kw: FakeFactor(m, s, **kw))
    return made


def golden_job(golden, name):
    """what tests/cases.py hands the host-built path: masked cellmap, filtered points, exclude set"""
    cfg, inp, exp = co.load_case(golden, name)
    fl = co.cfg_flags(cfg)
    cellmap, polymap, meta, inc = co.load_raster_inputs(cfg, inp)
    pk = inp["point_file"]
    points_rc = co.read_point_map(pk[0], pk[1], meta)
    exclude = set()
    if inc is not None:
        points_rc, exclude = co.generate_exclude_pairs(points_rc, inc)
    return dict(cellmap=cellmap, points_rc=points_rc, flags=cb.Flags.from_cfg(cfg), polymap=polymap,
                exclude_pairs=exclude, four_neighbors=fl["four_neighbors"], avg_res=fl["avg_res"]), exp


def assert_same_output(got, want, tol=1e-12):
    def close(a, b):
        a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
        assert a.shape == b.shape
        assert np.abs(a - b).max(initial=0.0) <= tol * max(1.0, np.abs(b).max(initial=0.0))
    close(got.resistances, want.resistances)
    assert got.num_solves == want.num_solves
    assert set(got.curmaps) == set(want.curmaps) and set(got.voltmaps) == set(want.voltmaps)
    for k in want.curmaps:
        close(got.curmaps[k], want.curmaps[k])
    for k in want.voltmaps:
        close(got.voltmaps[k], want.voltmaps[k])
    close(got.cum_curmap, want.cum_curmap)
    assert (got.max_curmap is None) == (want.max_curmap is None)
    if want.max_curmap is not None:
        close(got.max_curmap, want.max_curmap)


@pytest.mark.parametrize("i", range(1, 18))
def test_goldens_through_raster_pairwise(golden, cpu_device, i):
    job, exp = golden_job(golden, f"sgVerify{i}")
    got = cb.raster_pairwise(**job, solver=cb.CUDASolver())
    cases.check_raster_pairwise(got, exp, rel=1e-7)
    want, _ = cases.run_raster_pairwise(golden, f"sgVerify{i}", cb.CUDASolver())
    assert_same_output(got, want)
    ids = job["points_rc"][2]
    if len(ids) == len(np.unique(ids)):
        assert len(cpu_device) == 1                          # one whole-raster factor for the job
    else:
        u = np.unique(ids)
        pairs = [(a, b) for k, a in enumerate(u) for b in u[k + 1:]
                 if (a, b) not in job["exclude_pairs"] and (b, a) not in job["exclude_pairs"]]
        assert len(cpu_device) == len(pairs)                # one assembly per focal-region pair


def random_job(seed):
    rng = np.random.default_rng(seed)
    nr, nc = int(rng.integers(6, 13)), int(rng.integers(6, 13))
    g = island_raster(rng, nr, nc, holes=rng.choice([0.1, 0.3]))
    poly = island_polygons(rng, g) if rng.random() < 0.5 else None
    npts = int(rng.integers(3, 7))
    cells = rng.choice(nr * nc, size=npts, replace=False)
    rows, cols = cells % nr + 1, cells // nr + 1          # NODATA focal cells included
    ids = np.arange(1, npts + 1)
    if rng.random() < 0.35:
        ids[-1] = ids[0]                                   # a focal region: one assembly per pair
    order = np.argsort(ids, kind="stable")
    points_rc = (rows[order], cols[order], ids[order])
    u = np.unique(ids)
    exclude = {(int(u[0]), int(u[1]))} if rng.random() < 0.4 and len(u) >= 3 else set()
    keys = ["write_volt_maps", "write_cur_maps", "write_cum_cur_map_only", "write_max_cur_maps",
            "set_null_currents_to_nodata", "set_null_voltages_to_nodata", "log_transform_maps"]
    cfg = {k: str(bool(rng.random() < 0.5)) for k in keys}
    cfg.update(data_type="raster", scenario="pairwise")
    four, avg_res = bool(rng.random() < 0.5), bool(rng.random() < 0.3)
    return g, poly, points_rc, exclude, cfg, four, avg_res


class _Sink:
    def __init__(self):
        self.volt, self.cur = {}, {}

    def voltmap(self, key, grid):
        self.volt[key] = grid.copy()

    def curmap(self, key, grid):
        self.cur[key] = grid.copy()


@pytest.mark.parametrize("seed", range(40))
def test_random_multi_component_rasters_match_host_path(cpu_device, seed):
    g, poly, points_rc, exclude, cfg, four, avg_res = random_job(seed)
    flags = cb.Flags.from_cfg(cfg)
    ids = points_rc[2]
    if len(np.unique(ids)) < 2:
        return
    want = host_path(g, poly, points_rc, exclude, flags, four, avg_res)
    got = cb.raster_pairwise(g, points_rc, flags, polymap=poly, exclude_pairs=exclude, solver=cb.CUDASolver(),
                             four_neighbors=four, avg_res=avg_res)
    assert_same_output(got, want)
    sink = _Sink()
    streamed = cb.raster_pairwise(g, points_rc, flags, polymap=poly, exclude_pairs=exclude,
                                  solver=cb.CUDASolver(), four_neighbors=four, avg_res=avg_res, sink=sink)
    assert not streamed.curmaps and not streamed.voltmaps
    assert sink.cur.keys() == want.curmaps.keys() and sink.volt.keys() == want.voltmaps.keys()
    for k in want.curmaps:
        assert np.abs(sink.cur[k] - want.curmaps[k]).max() <= 1e-12 * max(1.0, np.abs(want.curmaps[k]).max())
    np.testing.assert_allclose(streamed.cum_curmap, got.cum_curmap, rtol=0, atol=0)


def host_path(g, poly, points_rc, exclude, flags, four, avg_res, solver=None):
    """the host-built path of tests/cases.py (graph.py front end + single_ground_all_pairs), for
    inputs that are not golden cases"""
    solver = solver or cb.CUDASolver()
    rr, cc_, ids = points_rc
    cellmap = g
    if len(ids) == len(np.unique(ids)):
        nodemap = graph.construct_node_map(cellmap, poly)
        G = graph.laplacian(graph.construct_graph(cellmap, nodemap, avg_res, four))
        prob = cb.GraphProblem(G, graph.connected_components(G), nodemap[rr - 1, cc_ - 1], ids, set(exclude),
                               nodemap, poly, cellmap, solver)
        return cb.single_ground_all_pairs(prob, flags)
    pts = list(dict.fromkeys(int(p) for p in ids))
    n = len(pts)
    R = -np.ones((n, n))
    merged = None
    for i in range(n):
        for j in range(i + 1, n):
            p1, p2 = pts[i], pts[j]
            if (p1, p2) in exclude or (p2, p1) in exclude:
                continue
            newpoly = co.create_new_polymap(cellmap, poly, points_rc, p1, p2)
            nodemap = graph.construct_node_map(cellmap, newpoly)
            G = graph.laplacian(graph.construct_graph(cellmap, nodemap, avg_res, four))
            x, y = int(np.nonzero(ids == p1)[0][0]), int(np.nonzero(ids == p2)[0][0])
            pn = np.array([nodemap[rr[x] - 1, cc_[x] - 1], nodemap[rr[y] - 1, cc_[y] - 1]])
            r = cb.single_ground_all_pairs(cb.GraphProblem(G, graph.connected_components(G), pn, np.array([p1, p2]),
                                                           set(), nodemap, newpoly, cellmap, solver), flags)
            R[i, j] = R[j, i] = r.resistances[1, 2]
            if merged is None:
                merged = r
                continue
            merged.voltmaps.update(r.voltmaps)
            merged.curmaps.update(r.curmaps)
            merged.cum_curmap = merged.cum_curmap + r.cum_curmap
            if merged.max_curmap is not None:
                merged.max_curmap = np.maximum(merged.max_curmap, r.max_curmap)
            merged.num_solves += r.num_solves
    np.fill_diagonal(R, 0.0)
    full = np.zeros((n + 1, n + 1))
    full[0, 1:] = full[1:, 0] = pts
    full[1:, 1:] = R
    merged.resistances = full
    return merged


def test_whole_raster_factor_requires_raster_mode(cpu_device):
    prob = cb.GraphProblem(None, [], np.array([1, 2]), np.array([1, 2]), coords=(np.array([1]), np.array([2])))
    with pytest.raises(ValueError):
        cb.solve(prob, cb.CUDASolver(), cb.Flags(is_raster=False), factor=object())


# ---- graph.create_pair_polymap ----------------------------------------------------------------------------
def _same_polymap(cellmap, polymap, points_rc, p1, p2):
    try:
        want = co.create_new_polymap(cellmap, polymap, points_rc, p1, p2)
    except NotImplementedError:
        with pytest.raises(ValueError):
            graph.create_pair_polymap(cellmap, polymap, points_rc, p1, p2)
        return
    got = graph.create_pair_polymap(cellmap, polymap, points_rc, p1, p2)
    assert np.array_equal(got, want)


@pytest.mark.parametrize("i", [5, 6, 8, 9, 10, 11])
def test_create_pair_polymap_on_goldens(golden, i):
    job, _ = golden_job(golden, f"sgVerify{i}")
    pts = list(dict.fromkeys(int(p) for p in job["points_rc"][2]))
    assert len(pts) < len(job["points_rc"][2]), "a focal-region case"
    for a in range(len(pts)):
        for b in range(a + 1, len(pts)):
            _same_polymap(job["cellmap"], job["polymap"], job["points_rc"], pts[a], pts[b])


@pytest.mark.parametrize("seed", range(30))
def test_create_pair_polymap_random(seed):
    rng = np.random.default_rng(seed)
    nr, nc = int(rng.integers(4, 10)), int(rng.integers(4, 10))
    g = rng.uniform(0.2, 2.0, (nr, nc))
    poly = None
    if rng.random() < 0.7:
        poly = np.zeros((nr, nc), dtype=np.int64)
        poly[rng.random((nr, nc)) < 0.25] = 1
        poly[rng.random((nr, nc)) < 0.15] = 4
    npts = int(rng.integers(3, 8))
    cells = rng.choice(nr * nc, size=npts, replace=False)
    ids = rng.integers(1, 4, npts)
    order = np.argsort(ids, kind="stable")
    points_rc = ((cells % nr + 1)[order], (cells // nr + 1)[order], ids[order])
    u = np.unique(ids)
    for a in range(len(u)):
        for b in range(a + 1, len(u)):
            _same_polymap(g, poly, points_rc, int(u[a]), int(u[b]))


def test_create_pair_polymap_single_overlap_raises():
    """a focal region with exactly one cell on a polygon: the reference's branch reads an undefined
    variable; the restatement refuses the input instead of guessing"""
    g = np.ones((3, 3))
    poly = np.zeros((3, 3), dtype=np.int64)
    poly[0, 0] = 2
    points_rc = (np.array([1, 3, 2]), np.array([1, 3, 2]), np.array([1, 1, 2]))
    with pytest.raises(ValueError):
        graph.create_pair_polymap(g, poly, points_rc, 1, 2)


# ---- on the device ------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("four", [False, True])
@pytest.mark.parametrize("polygons", [False, True])
@pytest.mark.parametrize("seed", [0, 1])
def test_device_components_of_raster_handles(seed, four, polygons):
    rng = np.random.default_rng(seed)
    g = island_raster(rng, 157 + 13 * seed, 121)
    g[rng.random(g.shape) < 0.2] = 0.0
    poly = island_polygons(rng, g) if polygons else None
    f, nodemap = cb.B200Factor.from_raster_polygons(g, poly, cb.CUDASolver(precond="jacobi"), four_neighbors=four)
    with f:
        lab, ncomp = f.components()
        lab2, ncomp2 = f.components()
    A = graph.laplacian(graph.construct_graph(np.where(g > 0, g, 0.0), nodemap, False, four))
    comps = graph.connected_components(A)
    assert ncomp == len(comps) > 3
    assert np.array_equal(lab, labels_of(comps, A.shape[0]))
    assert ncomp2 == ncomp and np.array_equal(lab2, lab)


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["double", "single"])
def test_device_components_of_a_network_handle(precision):
    """several disjoint power-law graphs, node ids shuffled so the components interleave"""
    blocks = [graph.power_law_laplacian(n, m=3, seed=s) for n, s in ((3000, 1), (500, 2), (40, 3), (1200, 4))]
    L = sp.block_diag(blocks + [sp.csr_matrix((1, 1))], format="csr")     # plus one isolated node
    perm = np.random.default_rng(5).permutation(L.shape[0])
    L = L[perm][:, perm].tocsr()
    L.sort_indices()
    solver = cb.CUDASolver(precond="jacobi", precision=precision, f32_compute=precision == "single")
    with cb.B200Factor(L, solver) as f:
        lab, ncomp = f.components()
        lab2, _ = f.components()
    comps = graph.connected_components(L)
    assert ncomp == len(comps) == 5
    assert np.array_equal(lab, labels_of(comps, L.shape[0])) and np.array_equal(lab2, lab)


@pytest.mark.gpu
def test_device_components_refused_with_grounds_applied():
    L = graph.synthetic_raster_laplacian(40, 30, seed=1)[0]
    with cb.B200Factor(L, cb.CUDASolver()) as f:
        mask = np.zeros(f.n, dtype=np.uint8)
        mask[3] = 1
        f.set_grounds(None, mask)
        with pytest.raises(cb.B200Error) as e:
            f.components()
        assert e.value.code == cb._lib.ERR_UNSUPPORTED
        f.set_grounds(None, None)
        lab, ncomp = f.components()
    assert ncomp == 1 and not lab.any()


@pytest.mark.gpu
@pytest.mark.parametrize("i", range(1, 18))
def test_goldens_through_raster_pairwise_on_device(golden, i):
    job, exp = golden_job(golden, f"sgVerify{i}")
    got = cb.raster_pairwise(**job, solver=cb.CUDASolver(rtol=1e-8))
    cases.check_raster_pairwise(got, exp, rel=1e-6)


@pytest.mark.gpu
@pytest.mark.parametrize("log_transform", [False, True])
def test_multi_component_raster_against_host_built_problem(log_transform):
    """~600 x 600 raster with islands and isolated cells, focal points in several components: the
    whole-raster factor against one factor per component (single_ground_all_pairs on the host-built
    problem)"""
    rng = np.random.default_rng(21)
    nr, nc = 600, 590
    g = 1.0 / rng.uniform(1.0, 10.0, (nr, nc))
    g[rng.random(g.shape) < 0.03] = 0.0                     # isolated cells and small holes
    g[:, 300] = 0.0                                         # three islands ...
    g[200, :] = 0.0
    g[450:470, 100:120] = 0.0
    g[455:465, 105:115] = 0.5                               # ... and a small one inside a frame of NODATA
    g[450:470, 100:120][[0, -1], :] = 0.0
    pts = [(20, 20), (150, 250), (100, 100), (400, 50), (550, 280), (300, 500), (590, 580), (460, 110), (464, 112)]
    rows = np.array([p[0] for p in pts]) + 1
    cols = np.array([p[1] for p in pts]) + 1
    ids = np.arange(1, len(pts) + 1)
    cfg = {"write_cur_maps": "True", "write_volt_maps": "True", "write_max_cur_maps": "True",
           "log_transform_maps": str(log_transform), "data_type": "raster", "scenario": "pairwise"}
    flags = cb.Flags.from_cfg(cfg)
    solver = cb.CUDASolver(rtol=1e-10)
    new = cb.raster_pairwise(g, (rows, cols, ids), flags, solver=solver)
    nodemap = graph.construct_node_map(np.where(g > 0, g, 0.0), None)
    G = graph.laplacian(graph.construct_graph(np.where(g > 0, g, 0.0), nodemap, False, False))
    comps = graph.connected_components(G)
    points = nodemap[rows - 1, cols - 1]
    lab = labels_of(comps, G.shape[0])
    assert len(np.unique(lab[points[points != 0] - 1])) >= 3
    old = cb.single_ground_all_pairs(cb.GraphProblem(G, comps, points, ids, set(), nodemap, None, g, solver), flags)
    print(f"\n[raster_pairwise] log={log_transform}: {new.num_solves} pairs, iterations whole-raster factor "
          f"{new.iterations}, per-component factors {old.iterations}")
    assert new.num_solves == old.num_solves > 0
    Rn, Ro = new.resistances[1:, 1:], old.resistances[1:, 1:]
    assert np.array_equal(Rn == -1, Ro == -1)
    ok = Ro > 0
    assert np.abs(Rn[ok] - Ro[ok]).max() <= 1e-9 * Ro[ok].max()
    scale = lambda m: np.abs(m).max()
    assert np.abs(new.cum_curmap - old.cum_curmap).max() <= 1e-6 * scale(old.cum_curmap)
    assert np.abs(new.max_curmap - old.max_curmap).max() <= 1e-6 * scale(old.max_curmap)
    cellcomp = np.where(nodemap > 0, lab[np.maximum(nodemap, 1) - 1], -1)
    pos = {int(i): k for k, i in enumerate(ids)}
    assert set(new.curmaps) == set(old.curmaps)
    for key in old.curmaps:
        outside = cellcomp != lab[points[pos[key[0]]] - 1]
        assert np.array_equal(new.curmaps[key][outside], old.curmaps[key][outside])
        assert np.array_equal(new.voltmaps[key][outside], old.voltmaps[key][outside])
        inside = ~outside
        assert np.abs(new.curmaps[key][inside] - old.curmaps[key][inside]).max() <= 1e-6 * scale(old.curmaps[key])
    # every column passes the residual gate (solve_pairs raises SolverResidualError otherwise); checked
    # here on the whole-raster factor directly
    f, _ = cb.B200Factor.from_raster_polygons(g, None, solver)
    with f:
        comp_of = lab[points - 1]
        src = [points[a] - 1 for a in range(len(pts)) for b in range(a + 1, len(pts)) if comp_of[a] == comp_of[b]]
        dst = [points[b] - 1 for a in range(len(pts)) for b in range(a + 1, len(pts)) if comp_of[a] == comp_of[b]]
        r = f.solve_pairs(src, dst)
    assert r["relres"].max() < 1e-4
