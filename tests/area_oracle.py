"""numpy restatement of the measurement areas (oc_areas_acc in include/optimal_crowds.h), independent of the library:
the even-odd membership rule in FP64 and the fixed summation order of the float sums (blocks of 256 agents, an xor
butterfly inside each warp of 32, the 8 warp sums in warp order, the block sums in block order)."""
import numpy as np

BLOCK, WARP = 256, 32


def _orient(ax, ay, bx, by, px, py):
    return (bx - ax) * (py - ay) - (by - ay) * (px - ax)


def inside(poly, x, y):
    """bool (N,): the even-odd rule for the polygon poly ((n, 2)) at the points (x, y); for every edge (a, b), b the
    vertex after a, when (a.y <= p.y) != (b.y <= p.y) the point toggles if (b.y > a.y) ? o(a,b,p) > 0 : o(a,b,p) < 0"""
    x, y = np.asarray(x, dtype=np.float64), np.asarray(y, dtype=np.float64)
    res = np.zeros(x.shape, dtype=bool)
    n = len(poly)
    with np.errstate(invalid="ignore"):
        for k in range(n):
            (ax, ay), (bx, by) = poly[k - 1], poly[k]
            cross = (ay <= y) != (by <= y)
            o = _orient(ax, ay, bx, by, x, y)
            res ^= cross & ((o > 0) if by > ay else (o < 0))
    return res


def fixed_order_sum(v):
    """the library's sum of the per-agent values v (N,): zero-padded to whole blocks, butterflies 16, 8, 4, 2, 1 in each
    warp, warp sums added in order from 0.0, block sums added in order from 0.0"""
    v = np.asarray(v, dtype=np.float64)
    nb = -(-len(v) // BLOCK)
    pad = np.zeros(nb * BLOCK)
    pad[:len(v)] = v
    w = pad.reshape(nb, BLOCK // WARP, WARP)
    lane = np.arange(WARP)
    for off in (16, 8, 4, 2, 1):
        w = w + w[:, :, lane ^ off]
    total = 0.0
    for b in range(nb):
        s = 0.0
        for k in range(BLOCK // WARP):
            s = s + w[b, k, 0]
        total = total + s
    return total


def measure(polys, x, y, vx, vy, status):
    """dict(count (A,) int, speed_sum, vx_sum, vy_sum (A,) float64) of one state: agents with status 1 inside each
    polygon; speeds sqrt(vx*vx + vy*vy)"""
    x, y, vx, vy = (np.asarray(a, dtype=np.float64) for a in (x, y, vx, vy))
    act = np.asarray(status) == 1
    with np.errstate(invalid="ignore", over="ignore"):
        s = np.sqrt(vx * vx + vy * vy)
    out = dict(count=[], speed_sum=[], vx_sum=[], vy_sum=[])
    for p in polys:
        m = act & inside(np.asarray(p, dtype=np.float64), x, y)
        out["count"].append(int(m.sum()))
        for k, a in (("speed_sum", s), ("vx_sum", vx), ("vy_sum", vy)):
            out[k].append(fixed_order_sum(np.where(m, a, 0.0)))
    return {k: np.array(v, dtype=np.int32 if k == "count" else np.float64) for k, v in out.items()}


def run_area_rows(polys, rows, exit_step, steps):
    """the rows of a run from its trajectory record (rows[k]: (N, 4) x, y, vx, vy after k steps) and exit steps: row k
    measures rows[k] with the agents that had not left before step k"""
    exit_step = np.asarray(exit_step)
    out = dict(count=[], speed_sum=[], vx_sum=[], vy_sum=[])
    for k in range(steps):
        r = rows[k]
        st = ((exit_step < 0) | (exit_step >= k)).astype(np.uint8)
        m = measure(polys, r[:, 0], r[:, 1], r[:, 2], r[:, 3], st)
        for key in out:
            out[key].append(m[key])
    A = len(polys)
    return {k: np.array(v, dtype=np.int32 if k == "count" else np.float64).reshape(steps, A) for k, v in out.items()}
