"""Python restatement of the Voronoi measures of measurement areas (oc_voronoi_acc in include/optimal_crowds.h),
independent of the library apart from its inputs: the areas' triangles (simulations.voronoi_triangles, whose own
properties tests/test_cpu_voronoi.py checks) and |A|.  Every operation is one IEEE double operation, as the header
writes it; the float sums use the measurement areas' fixed order (area_oracle.fixed_order_sum).

  1. Generators: status 1 and finite x and y.
  2. Agent i starts from the polygon (x_i + r*cos(2*pi*k/n), y_i + r*sin(2*pi*k/n)), k = 0..n-1.
  3. A Sutherland-Hodgman pass keeps s <= 0 (each vertex's s once; the crossing point a + t*(b - a), t = sa / (sa - sb));
     fewer than 3 vertices is empty, more than 64 overflows (area NaN).
  4. The cell: clipped by -x, x - L, -y, y - H, then by every other generator j in ascending index with
     dx*dx + dy*dy <= (2r)*(2r) and (dx, dy) != (0, 0), s = dx*(p.x - mx) + dy*(p.y - my).
  5. |V| = 0.5 * sum(x_k*y_{k+1} - x_{k+1}*y_k) from 0.0.
  6. w = sum over the area's triangles whose bounding box the square [x +- r] x [y +- r] meets of |V clipped by
     -o(a,b,p), -o(b,c,p), -o(c,a,p)|; NaN for an overflowed cell that meets one.
  7. Terms w/|V|, w*s, w*vx, w*vy, w, all +0.0 for non-generators, |V| <= 0 and w == 0.
  8. The five fixed-order sums over the agents, divided by |A|: density, speed, velocity (vx, vy), covered."""
import math

import numpy as np

from area_oracle import fixed_order_sum

CAP = 64


def clip(P, s):
    """one Sutherland-Hodgman pass of the polygon P (list of (x, y); [] empty, None overflowed) keeping s(p) <= 0"""
    if P is None or len(P) < 3:
        return P if P is None else []
    n = len(P)
    sv = [s(p) for p in P]
    out = []
    for k in range(n):
        a, b = P[k], P[(k + 1) % n]
        sa, sb = sv[k], sv[(k + 1) % n]
        if sa <= 0:
            out.append(a)
        if (sa <= 0) != (sb <= 0):
            t = sa / (sa - sb)
            out.append((a[0] + t * (b[0] - a[0]), a[1] + t * (b[1] - a[1])))
    if len(out) > CAP:
        return None
    return out if len(out) >= 3 else []


def area(P):
    """the shoelace area of rule 5 (NaN for an overflowed polygon)"""
    if P is None:
        return math.nan
    s = 0.0
    n = len(P)
    for k in range(n):
        a, b = P[k], P[(k + 1) % n]
        s += a[0] * b[1] - b[0] * a[1]
    return 0.5 * s


def ring(cutoff, edges):
    k = np.arange(edges)
    return cutoff * np.cos(2 * np.pi * k / edges), cutoff * np.sin(2 * np.pi * k / edges)


def generators(x, y, status):
    x, y = np.asarray(x, dtype=np.float64), np.asarray(y, dtype=np.float64)
    return (np.asarray(status) == 1) & np.isfinite(x) & np.isfinite(y)


def cell(i, x, y, gen, L, H, cutoff, ox, oy):
    """the cell of generator i (list of vertices, [] empty, None overflowed)"""
    xi, yi = float(x[i]), float(y[i])
    P = [(xi + float(a), yi + float(b)) for a, b in zip(ox, oy)]
    P = clip(P, lambda p: -p[0])
    P = clip(P, lambda p: p[0] - L)
    P = clip(P, lambda p: -p[1])
    P = clip(P, lambda p: p[1] - H)
    with np.errstate(over="ignore", invalid="ignore"):
        dx, dy = x - xi, y - yi
        near = gen & (dx * dx + dy * dy <= (2.0 * cutoff) * (2.0 * cutoff)) & ~((dx == 0) & (dy == 0))
    for j in np.nonzero(near)[0]:                                # ascending index
        if not P:
            break
        xj, yj = float(x[j]), float(y[j])
        ddx, ddy = xj - xi, yj - yi
        mx, my = 0.5 * (xi + xj), 0.5 * (yi + yj)
        P = clip(P, lambda p: ddx * (p[0] - mx) + ddy * (p[1] - my))
    return P


def _orient_clip(P, a, b):
    ax, ay, bx, by = a[0], a[1], b[0], b[1]
    return clip(P, lambda p: -((bx - ax) * (p[1] - ay) - (by - ay) * (p[0] - ax)))


def measure(tris, areas_abs, L, H, cutoff, edges, x, y, vx, vy, status):
    """dict(density, speed, covered (A,), velocity (A, 2)) of one state; tris: per area an (t, 3, 2) array of its
    counter-clockwise triangles; areas_abs: (A,) |A|"""
    x, y, vx, vy = (np.asarray(a, dtype=np.float64) for a in (x, y, vx, vy))
    N, A, r = len(x), len(tris), float(cutoff)
    gen = generators(x, y, status)
    ox, oy = ring(cutoff, edges)
    boxes = [np.stack([t[:, :, 0].min(1), t[:, :, 0].max(1), t[:, :, 1].min(1), t[:, :, 1].max(1)], axis=1)
             for t in tris]
    terms = np.zeros((A, 5, N))
    for i in np.nonzero(gen)[0]:
        xl, xh, yl, yh = x[i] - r, x[i] + r, y[i] - r, y[i] + r
        meets = [np.nonzero((xl <= b[:, 1]) & (xh >= b[:, 0]) & (yl <= b[:, 3]) & (yh >= b[:, 2]))[0] for b in boxes]
        if not any(len(m) for m in meets):
            continue
        V = cell(i, x, y, gen, L, H, cutoff, ox, oy)
        vol = area(V)
        if not (vol > 0) and V is not None:
            continue
        s = math.sqrt(vx[i] * vx[i] + vy[i] * vy[i])
        for a in range(A):
            w = 0.0
            for t in meets[a]:
                if V is None:
                    w = math.nan
                    break
                pa, pb, pc = tris[a][t]
                w += area(_orient_clip(_orient_clip(_orient_clip(V, pa, pb), pb, pc), pc, pa))
            if w != 0.0:
                terms[a, :, i] = (w / vol, w * s, w * vx[i], w * vy[i], w)
    sums = np.array([[fixed_order_sum(terms[a, q]) for q in range(5)] for a in range(A)]).reshape(A, 5)
    out = sums / np.asarray(areas_abs, dtype=np.float64)[:, None]
    return dict(density=out[:, 0], speed=out[:, 1], velocity=out[:, 2:4], covered=out[:, 4])


def run_rows(tris, areas_abs, L, H, cutoff, edges, rows, exit_step, steps):
    """the Voronoi rows of a run from its trajectory record (rows[k]: (N, 4) x, y, vx, vy after k steps) and exit steps:
    row k measures rows[k] with the agents that had not left before step k"""
    exit_step = np.asarray(exit_step)
    out = dict(density=[], speed=[], velocity=[], covered=[])
    for k in range(steps):
        r = rows[k]
        st = ((exit_step < 0) | (exit_step >= k)).astype(np.uint8)
        m = measure(tris, areas_abs, L, H, cutoff, edges, r[:, 0], r[:, 1], r[:, 2], r[:, 3], st)
        for key in out:
            out[key].append(m[key])
    return {k: np.array(v, dtype=np.float64) for k, v in out.items()}
