"""NumPy restatement of the spatially regularised spectrum fit (definition in csrc/met2_spatial.cu, DESIGN.md §10b).

Neighbour table and colours by explicit loops over the voxels, each block update as one Lawson-Hanson solve
(oracle/met2_oracle.py: lh_nnls) of the stacked system A = [D; sqrt(lam) L; sqrt(mu n_v) I], b = [y; 0; sqrt(mu n_v) p],
and the joint objective J.  Spectra are in the reference's normalised units (fsol / sig[0])."""
import numpy as np

import met2_oracle as O

# face order of the neighbour table: -x, +x, -y, +y, -z, +z
FACES = ((-1, 0, 0), (1, 0, 0), (0, -1, 0), (0, 1, 0), (0, 0, -1), (0, 0, 1))


def neighbours(flat, shape, fitted):
    """flat[V]: C-order indices of the masked voxels in a volume of `shape`; fitted[V]: bool.  Returns nbr[V, 6]
    (positions in 0..V-1 of the fitted face neighbours, -1 = none; all -1 for a voxel that is not fitted) and the two
    colour lists (positions of the fitted voxels with (i + j + k) % 2 == 0, == 1), ascending."""
    nx, ny, nz = shape
    where = {}
    for i, f in enumerate(flat):
        if fitted[i]:
            where[int(f)] = i
    V = len(flat)
    nbr = np.full((V, 6), -1, dtype=np.int32)
    colours = ([], [])
    for i, f in enumerate(flat):
        if not fitted[i]:
            continue
        a, r = divmod(int(f), ny * nz)
        b, c = divmod(r, nz)
        for k, (dx, dy, dz) in enumerate(FACES):
            q = (a + dx, b + dy, c + dz)
            if 0 <= q[0] < nx and 0 <= q[1] < ny and 0 <= q[2] < nz:
                nbr[i, k] = where.get((q[0] * ny + q[1]) * nz + q[2], -1)
        colours[(a + b + c) % 2].append(i)
    return nbr, tuple(np.array(c, dtype=np.int32) for c in colours)


def block_update(D, y, L, lam, mu, p, nv):
    """argmin_{x >= 0} ||D x - y||^2 + lam ||L x||^2 + mu nv ||x - p||^2 by Lawson-Hanson on the stacked system.
    Returns (x, mode) with mode 3 when itmax was reached."""
    n = D.shape[1]
    w = mu * nv
    A = np.concatenate((D, np.sqrt(lam) * L, np.sqrt(w) * np.eye(n)))
    b = np.concatenate((y, np.zeros(n), np.sqrt(w) * p))
    x, _, mode = O.lh_nnls(A, b)
    return x, mode


def half_sweep(x, vox, Y, Dv, lam, L, nbr, mu):
    """Block updates of the voxels `vox` (one colour) with the others held fixed.  Y[V, nTE] normalised signals,
    Dv(v) -> the dictionary D_{a_v} [nTE, nT2], lam[V].  Returns (new x, positions whose solve hit itmax)."""
    x = np.array(x, dtype=np.float64, copy=True)
    itmax = []
    for v in vox:
        q = nbr[v][nbr[v] >= 0]
        p = x[q].mean(axis=0) if len(q) else np.zeros(x.shape[1])
        x[v], mode = block_update(Dv(v), Y[v], L, lam[v], mu, p, len(q))
        if mode == 3:
            itmax.append(int(v))
    return x, itmax


def sweeps(x0, colours, Y, Dv, lam, L, nbr, mu, n_sweeps):
    """n_sweeps red-black sweeps from x0; returns (x, [x after every half-sweep])."""
    x, trace = x0, []
    for _ in range(n_sweeps):
        for vox in colours:
            x, _ = half_sweep(x, vox, Y, Dv, lam, L, nbr, mu)
            trace.append(x)
    return x, trace


def objective(x, fitted, Y, Dv, lam, L, nbr, mu):
    """J(x) over the fitted voxels; every edge counted once (the +x, +y and +z faces)."""
    J = 0.0
    for v in np.nonzero(fitted)[0]:
        r = Dv(v) @ x[v] - Y[v]
        J += r @ r + lam[v] * np.sum((L @ x[v]) ** 2)
        for k in (1, 3, 5):
            q = nbr[v, k]
            if q >= 0:
                d = x[v] - x[q]
                J += mu * (d @ d)
    return J
