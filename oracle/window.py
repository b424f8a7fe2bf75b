"""TEST INFRASTRUCTURE -- numpy restatement of the pruning bound of the range-image window searches (csrc/window.cuh:
make_eval_geom and the stop rule of window_search).  NOT product code.

A query at range rq stops growing its window at half-sizes (dr, dc) once the squared distance it still has to beat lies
below

    stop_bound(rq, s2) = f32(f32(f32(rq * rq) * f32(1 - 2e-3)) * s2),   s2 = min(row_s2[dr + 1], col_s2[dc + 1]),

so the search is exact when every valid pixel k or more rows (columns) away from the query is at a cham_d of at least
stop_bound(rq, row_s2[k]) (col_s2[k]).  eval_geom gives the tables in the device's order of operations; tau is their
absolute angular slack, margin their relative one on the squared distance (DESIGN.md §4, "Window-pruned chamfer").
"""
import math

import numpy as np

F32 = np.float32
KEVR = 48              # kEvR: largest window half-size held in the tables
TAU = 1e-6             # kEvTau: absolute angular slack (rad)
MARGIN = 2e-3          # relative margin on the squared distance


def eval_geom(H, W, hfov, vmax, vmin, tau=TAU):
    """-> (row_s2, col_s2), (KEVR + 2,) f32 each: sin^2 of the smallest angle, less tau, between the query's ray and any
    ray >= k rows / >= k columns (circularly) away."""
    dalt = (vmax - vmin) / float(H - 1)
    daz = hfov / float(W)
    cmin = math.cos(max(abs(vmax), abs(vmin)))
    half_pi = 1.57079632679489661923
    row = np.empty(KEVR + 2, F32)
    col = np.empty(KEVR + 2, F32)
    for k in range(KEVR + 2):
        tr = max(0.0, k * dalt - tau)
        row[k] = F32(1.0) if tr >= half_pi else F32(math.sin(tr) * math.sin(tr))
        az = min(k * daz, 3.14159265358979323846)
        sh = cmin * math.sin(az / 2)
        t = max(0.0, 2.0 * math.asin(min(sh, 1.0)) - tau)
        col[k] = F32(1.0) if t >= half_pi else F32(math.sin(t) * math.sin(t))
    return row, col


def stop_bound(rq, s2, margin=MARGIN):
    """The squared distance below which window_search stops, for queries at f32 ranges rq and table entries s2."""
    rq = np.asarray(rq, F32)
    r2 = ((rq * rq).astype(F32) * (F32(1.0) - F32(margin))).astype(F32)
    return (r2 * np.asarray(s2, F32)).astype(F32)
