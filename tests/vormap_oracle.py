"""Python restatement of the Voronoi maps (oc_vormap_acc in include/optimal_crowds.h), independent of the library apart
from its inputs.  The cells are tests/voronoi_oracle.py's (rules 1-5 of oc_voronoi_acc); the owner of a node is found
by a brute-force search over all generators in ascending index, with no bins.  Every operation is one IEEE double
operation, as the header writes it.

  2. Nodes p = (X[ix], Y[iy]); nodes with Vglobal < 0 are walls, never covered.
  3. Owner: the generator with the smallest d2 = (X-x)*(X-x) + (Y-y)*(Y-y) among those with d2 <= r*r, the lowest index
     on ties; none: uncovered.
  4. p must satisfy o(a_k, a_{k+1}, p) >= 0 for every edge of the owner's cut-off polygon, else uncovered.
  5. Terms 1/|V|, s = sqrt(vx*vx + vy*vy), vx, vy; |V| <= 0 uncovered; |V| NaN covered with NaN terms.
  6. density_sum += rho, density_max = np.maximum(density_max, rho) (rho = 0 when uncovered), covered += 1, then the
     sums of s, vx and vy -- at covered nodes only, density_max everywhere."""
import math

import numpy as np

from voronoi_oracle import area, cell, generators, ring

BLOCK = 64   # generators per vectorised pass of the owner search


def owners(X, Y, x, y, gen, cutoff):
    """(Ny, Nx) int64: the owner of every node by rule 3 (-1: none), brute force over all generators"""
    XX, YY = np.meshgrid(np.asarray(X, dtype=np.float64), np.asarray(Y, dtype=np.float64))
    XX, YY = XX.ravel(), YY.ravel()
    best = np.full(XX.shape, np.inf)
    own = np.full(XX.shape, -1, dtype=np.int64)
    rr = cutoff * cutoff
    idx = np.nonzero(gen)[0]
    cols = np.arange(XX.size)
    for b in range(0, len(idx), BLOCK):
        js = idx[b:b + BLOCK]
        with np.errstate(over="ignore", invalid="ignore"):
            dx = XX[None, :] - x[js][:, None]
            dy = YY[None, :] - y[js][:, None]
            d2 = dx * dx + dy * dy
        d2 = np.where(d2 <= rr, d2, np.inf)
        k = np.argmin(d2, axis=0)                      # the first minimum: the lowest index of the block
        dk = d2[k, cols]
        take = dk < best                                # strict: an earlier block's generator keeps its ties
        best[take] = dk[take]
        own[take] = js[k[take]]
    return own.reshape(len(Y), len(X))


def frame(X, Y, Vg, L, H, cutoff, edges, x, y, vx, vy, status):
    """the terms of one frame: dict(covered (Ny, Nx) bool, rho, s, vx, vy (Ny, Nx) float64, owner (Ny, Nx))"""
    x, y, vx, vy = (np.asarray(a, dtype=np.float64) for a in (x, y, vx, vy))
    X, Y = np.asarray(X, dtype=np.float64), np.asarray(Y, dtype=np.float64)
    gen = generators(x, y, status)
    ox, oy = ring(cutoff, edges)
    own = owners(X, Y, x, y, gen, cutoff)
    own[np.asarray(Vg) < 0] = -1
    XX, YY = np.meshgrid(X, Y)
    iy, ix = np.nonzero(own >= 0)
    i = own[iy, ix]
    px, py = XX[iy, ix], YY[iy, ix]
    xi, yi = x[i], y[i]
    ok = np.ones(len(i), dtype=bool)
    for k in range(edges):
        k1 = (k + 1) % edges
        ax, ay, bx, by = xi + ox[k], yi + oy[k], xi + ox[k1], yi + oy[k1]
        ok &= (bx - ax) * (py - ay) - (by - ay) * (px - ax) >= 0
    iy, ix, i = iy[ok], ix[ok], i[ok]
    vol = {j: area(cell(j, x, y, gen, L, H, cutoff, ox, oy)) for j in np.unique(i)}
    shape = own.shape
    out = dict(covered=np.zeros(shape, dtype=bool), rho=np.zeros(shape), s=np.zeros(shape), vx=np.zeros(shape),
               vy=np.zeros(shape), owner=np.full(shape, -1, dtype=np.int64))
    for a, b, j in zip(iy, ix, i):
        v = vol[j]
        if math.isnan(v):
            out["covered"][a, b] = True
            out["rho"][a, b] = out["s"][a, b] = out["vx"][a, b] = out["vy"][a, b] = math.nan
        elif v > 0:
            out["covered"][a, b] = True
            u, w = vx[j], vy[j]
            out["rho"][a, b] = 1.0 / v
            out["s"][a, b] = math.sqrt(u * u + w * w)
            out["vx"][a, b], out["vy"][a, b] = u, w
        else:
            continue
        out["owner"][a, b] = j
    return out


def empty(shape):
    """the accumulators of rule 6 before any frame (zeros)"""
    return dict(density_sum=np.zeros(shape), density_max=np.zeros(shape), covered=np.zeros(shape, dtype=np.int32),
                speed_sum=np.zeros(shape), vx_sum=np.zeros(shape), vy_sum=np.zeros(shape), frames=0)


def add(acc, t):
    """rule 6: one frame's terms t (frame()) added to acc in place"""
    c = t["covered"]
    acc["density_sum"][c] = acc["density_sum"][c] + t["rho"][c]
    acc["density_max"] = np.maximum(acc["density_max"], np.where(c, t["rho"], 0.0))
    acc["covered"][c] += 1
    for k, q in (("speed_sum", "s"), ("vx_sum", "vx"), ("vy_sum", "vy")):
        acc[k][c] = acc[k][c] + t[q][c]
    acc["frames"] += 1
    return acc


def run_maps(X, Y, Vg, L, H, cutoff, edges, every, rows, exit_step, steps):
    """the maps of a run from its trajectory record (rows[k]: (N, 4) x, y, vx, vy after k steps) and exit steps: a frame
    of rows[k], with the agents that had not left before step k, for every k < steps that is a multiple of every"""
    exit_step = np.asarray(exit_step)
    acc = empty((len(Y), len(X)))
    for k in range(0, steps, every):
        r = np.asarray(rows[k], dtype=np.float64)
        st = ((exit_step < 0) | (exit_step >= k)).astype(np.uint8)
        add(acc, frame(X, Y, Vg, L, H, cutoff, edges, r[:, 0], r[:, 1], r[:, 2], r[:, 3], st))
    return acc
