"""raster_pairwise end to end against the host-built path it replaces, on one GPU.

    python profiles/raster_pairwise_e2e.py [--size 3163] [--points 16] [--repeats 2] [--out DIR]

Two rasters: the bench's (graph.synthetic_raster_laplacian(size, size, seed=42), every cell a node) and
the same conductances with 2 % NODATA cells plus two NODATA lines that cut it into four islands.
Focal points: `--points` cells from graph.focal_nodes(..., seed=7) (valid cells only), all pairs;
cumulative and max current maps on.

  old   graph.py front end (node map, construct_graph, laplacian, connected_components) + GraphProblem
        + single_ground_all_pairs (a host submatrix and a fresh handle per component)
  new   circuitscape_b200.raster_pairwise (device assembly, cs_b200_components, one whole-raster factor)

The two alternate inside one process; then one more run of the new path broken into assembly,
components, solves and maps (each ends in a device synchronise: every step returns host data).
Prints one JSON object and writes it to DIR/raster_pairwise_e2e.json."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import circuitscape_b200 as cb                      # noqa: E402
from circuitscape_b200 import core, graph          # noqa: E402
from circuitscape_b200 import solver as S          # noqa: E402


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = (s.strip() for s in q.split(","))
        return dict(name=name, power_limit=power, max_sm_clock=clock)
    except Exception as e:                          # the numbers stay valid without it, but say so
        return dict(error=str(e))


def rasters(size):
    _, g = graph.synthetic_raster_laplacian(size, size, seed=42)
    g2 = g.copy()
    rng = np.random.default_rng(1)
    g2[rng.random(g2.shape) < 0.02] = 0.0
    g2[:, size // 3] = 0.0
    g2[2 * size // 3, :] = 0.0
    return {"full": g, "nodata_islands": g2}


def focal_points(g, count):
    valid = np.flatnonzero((g > 0).ravel(order="F"))
    cells = valid[graph.focal_nodes(len(valid), count, seed=7)]
    rows, cols = cells % g.shape[0] + 1, cells // g.shape[0] + 1
    return rows, cols, np.arange(1, count + 1)


def old_path(g, points_rc, flags, solver):
    rr, cc_, ids = points_rc
    t0 = time.perf_counter()
    nodemap = graph.construct_node_map(g, None)
    G = graph.laplacian(graph.construct_graph(g, nodemap, False, False))
    comps = graph.connected_components(G)
    prob = cb.GraphProblem(G, comps, nodemap[rr - 1, cc_ - 1], ids, set(), nodemap, None, g, solver)
    t1 = time.perf_counter()
    out = cb.single_ground_all_pairs(prob, flags)
    t2 = time.perf_counter()
    return out, dict(front_end_s=t1 - t0, driver_s=t2 - t1, total_s=t2 - t0)


def new_path(g, points_rc, flags, solver):
    t0 = time.perf_counter()
    out = cb.raster_pairwise(g, points_rc, flags, solver=solver)
    return out, dict(total_s=time.perf_counter() - t0)


def new_path_phases(g, points_rc, flags, solver):
    rr, cc_, ids = points_rc
    ph = {}
    t = time.perf_counter()
    f, nodemap = S.B200Factor.from_raster_polygons(g, None, solver)
    ph["assembly_and_setup_s"] = time.perf_counter() - t
    with f:
        t = time.perf_counter()
        labels, ncomp = f.components()
        ph["components_s"] = time.perf_counter() - t
        t = time.perf_counter()
        points = nodemap[rr - 1, cc_ - 1]
        prob = cb.GraphProblem(None, core._focal_components(f, points), points, ids, set(), nodemap, None, g, solver)
        ph["component_lists_s"] = time.perf_counter() - t
        maps = {}
        inner = core._add_whole_raster_currents

        def timed(*a, **kw):
            t_ = time.perf_counter()
            inner(*a, **kw)
            maps["s"] = time.perf_counter() - t_
        core._add_whole_raster_currents = timed
        try:
            t = time.perf_counter()
            out = core.solve(prob, solver, flags, factor=f)
            total = time.perf_counter() - t
        finally:
            core._add_whole_raster_currents = inner
        ph["maps_s"] = maps.get("s", 0.0)
        ph["solves_s"] = total - ph["maps_s"]
        # the component kernel alone, on the resident handle (labels back to the host included)
        reps = 5
        t = time.perf_counter()
        for _ in range(reps):
            f.components()
        ph["components_warm_s"] = (time.perf_counter() - t) / reps
        ph.update(n=int(f.n), ncomp=int(ncomp),
                  focal_components=len(prob.cc), num_solves=out.num_solves, iterations=out.iterations)
    return ph


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--size", type=int, default=3163)
    ap.add_argument("--points", type=int, default=16)
    ap.add_argument("--repeats", type=int, default=2)
    ap.add_argument("--out", default=".", help="directory the JSON result is written to")
    a = ap.parse_args()
    flags = cb.Flags(is_raster=True, outputflags=cb.OutputFlags(write_cum_cur_map_only=True, write_max_cur_maps=True))
    solver = cb.CUDASolver()
    res = dict(card=card(), size=a.size, points=a.points, rtol=solver.rtol, cases={})
    for name, g in rasters(a.size).items():
        pts = focal_points(g, a.points)
        runs = {"old": [], "new": []}
        outs = {}
        for _ in range(a.repeats):
            for which, fn in (("old", old_path), ("new", new_path)):
                o, t = fn(g, pts, flags, solver)
                runs[which].append(t)
                outs[which] = o
                print(f"[{name}] {which}: {t}", flush=True)
        o, n = outs["old"], outs["new"]
        ok = o.resistances[1:, 1:] > 0
        dR = float((np.abs(n.resistances[1:, 1:] - o.resistances[1:, 1:])[ok] / o.resistances[1:, 1:][ok]).max())
        dcum = float(np.abs(n.cum_curmap - o.cum_curmap).max() / np.abs(o.cum_curmap).max())
        dmax = float(np.abs(n.max_curmap - o.max_curmap).max() / np.abs(o.max_curmap).max())
        ph = new_path_phases(g, pts, flags, solver)
        res["cases"][name] = dict(runs=runs, num_solves=n.num_solves, iterations_new=n.iterations,
                                  iterations_old=o.iterations, max_rel_dR=dR, max_rel_dcum=dcum, max_rel_dmax=dmax,
                                  new_phases=ph)
        print(f"[{name}] phases {ph}  max rel dR {dR:.2e}  dcum {dcum:.2e}  dmax {dmax:.2e}", flush=True)
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "raster_pairwise_e2e.json"), "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
