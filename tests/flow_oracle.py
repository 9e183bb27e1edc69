"""Reference rules of the flow statistics (test infrastructure only; the product package never imports this module).

Counting rule of the measurement lines (``simulation(..., lines=...)``, ``lines_count_kernel``).  With the orientation

    o(u, v, w) = (v.x - u.x) * (w.y - u.y) - (v.y - u.y) * (w.x - u.x)

evaluated in that order in float64 (numpy does not contract a*b - c*d into an FMA), and a line with endpoints a, b: an
agent inside at the start of step k that moves from p (its position before the step) to q (its position after it, also
in the step in which it leaves) crosses the line when

    (o(a, b, p) > 0) != (o(a, b, q) > 0)   and   (o(p, q, a) > 0) != (o(p, q, b) > 0).

The crossing is ``to_left`` when o(a, b, q) > 0 and ``to_right`` otherwise.  A point exactly on the line (o == 0) is on
the right side, so a move that ends on the line from the left counts to the right, a move from the line to the left
counts to the left, and a move along the line never counts.  A NaN compares false: a NaN position never crosses.

Velocity maps of a density frame (``density_stats=dict(velocity=True)``).  Agent i's weight at a node is the value the
density frame adds for it, w_i = ocm_exp(-r^2 / (2 sigma^2)) / C.  The C oracle ``oco_density`` of that agent alone is
exactly w_i (0.0 + w_i == w_i) with walls at 0, so the maps are built from single-agent oracle frames:
vx_f = sum_i w_i * vx_i, vy_f = sum_i w_i * vy_i, speed_f = sum_i w_i * sqrt(vx_i^2 + vy_i^2) in agent order from 0.0,
then 0 on walls.  Agents outside the device kernel's culling radius have w_i == 0 and add +-0, which leaves every sum
unchanged, so the unculled sum here equals the culled one bit for bit (finite velocities).
"""
from __future__ import annotations

import numpy as np


def orient(ux, uy, vx, vy, wx, wy):
    return (vx - ux) * (wy - uy) - (vy - uy) * (wx - ux)


def line_crossings(lines, p, q, inside):
    """crossings of one step: lines (L, 4) of (x0, y0, x1, y1); p, q (N, 2) positions before / after the step; inside (N,)
    bool, the agents inside at the start of the step.  -> (to_left, to_right): int32 (L,) counts"""
    lines = np.asarray(lines, dtype=np.float64).reshape(-1, 4)
    p, q = np.asarray(p, dtype=np.float64).reshape(-1, 2), np.asarray(q, dtype=np.float64).reshape(-1, 2)
    inside = np.asarray(inside, dtype=bool)
    px, py, qx, qy = p[inside, 0], p[inside, 1], q[inside, 0], q[inside, 1]
    left = np.zeros(len(lines), dtype=np.int32)
    right = np.zeros(len(lines), dtype=np.int32)
    for l, (ax, ay, bx, by) in enumerate(lines):
        sp = orient(ax, ay, bx, by, px, py) > 0
        sq = orient(ax, ay, bx, by, qx, qy) > 0
        cross = (sp != sq) & ((orient(px, py, qx, qy, ax, ay) > 0) != (orient(px, py, qx, qy, bx, by) > 0))
        left[l] = np.count_nonzero(cross & sq)
        right[l] = np.count_nonzero(cross & ~sq)
    return left, right


def run_line_counts(lines, rows, exit_step, steps):
    """the counts of a run from its trajectory record: rows[k] (N, >=2) = state after k steps, exit_step[i] = step in
    which agent i left (-1: still inside).  -> (to_left, to_right): int32 (steps, L)"""
    exit_step = np.asarray(exit_step)
    L = len(np.asarray(lines).reshape(-1, 4))
    left = np.zeros((steps, L), dtype=np.int32)
    right = np.zeros((steps, L), dtype=np.int32)
    for k in range(steps):
        inside = (exit_step < 0) | (exit_step >= k)
        left[k], right[k] = line_crossings(lines, rows[k][:, :2], rows[k + 1][:, :2], inside)
    return left, right


def velocity_frame(X, Y, Vglobal, x, y, vx, vy, status, sigma):
    """(vx_f, vy_f, speed_f): (Ny, Nx) velocity maps of one density frame, from single-agent frames of the C oracle"""
    from oracle import cpu_oracle as co
    shape = (len(Y), len(X))
    fu, fv, fs = np.zeros(shape), np.zeros(shape), np.zeros(shape)
    one = np.ones(1, dtype=np.uint8)
    for i in range(len(x)):
        if not status[i]:
            continue
        w = co.density(X, Y, Vglobal, x[i:i + 1], y[i:i + 1], one, sigma)
        u, v = float(vx[i]), float(vy[i])
        s = np.sqrt(np.float64(u) * u + np.float64(v) * v)
        fu = fu + w * u
        fv = fv + w * v
        fs = fs + w * s
    wall = np.asarray(Vglobal) < 0
    for f in (fu, fv, fs):
        f[wall] = 0.0
    return fu, fv, fs
