"""The NumPy restatement of the spatially regularised fit (tests/spatial_oracle.py) checked on its own: neighbour
table and colours by hand, the point problem at mu = 0, monotone J, independence of the voxel order."""
import numpy as np

import met2_oracle as O
import spatial_oracle as S


def test_neighbour_table_by_hand():
    # 3 x 3 x 2 volume, masked everywhere but (1, 1, 0) and (2, 2, 1); (0, 2, 1), (1, 2, 0) and (2, 1, 0) are masked
    # but not fitted, which leaves (0, 2, 0) one neighbour and (2, 2, 0) none
    shape = (3, 3, 2)
    mask = np.ones(shape, dtype=bool)
    mask[1, 1, 0] = mask[2, 2, 1] = False
    flat = np.nonzero(mask.ravel())[0]
    fitted = np.ones(len(flat), dtype=bool)
    pos = {int(f): i for i, f in enumerate(flat)}
    at = lambda i, j, k: pos[(i * 3 + j) * 2 + k]
    for ijk in ((0, 2, 1), (1, 2, 0), (2, 1, 0)):
        fitted[at(*ijk)] = False
    nbr, (c0, c1) = S.neighbours(flat, shape, fitted)
    #                     -x            +x            -y            +y            -z            +z
    assert list(nbr[at(0, 0, 0)]) == [-1, at(1, 0, 0), -1, at(0, 1, 0), -1, at(0, 0, 1)]
    assert list(nbr[at(1, 0, 1)]) == [at(0, 0, 1), at(2, 0, 1), -1, at(1, 1, 1), at(1, 0, 0), -1]
    assert list(nbr[at(0, 2, 0)]) == [-1, -1, at(0, 1, 0), -1, -1, -1]          # (1,2,0) and (0,2,1) not fitted
    assert list(nbr[at(1, 1, 1)]) == [at(0, 1, 1), at(2, 1, 1), at(1, 0, 1), at(1, 2, 1), -1, -1]   # (1,1,0) masked
    assert list(nbr[at(2, 2, 0)]) == [-1] * 6                                    # isolated
    for ijk in ((0, 2, 1), (1, 2, 0), (2, 1, 0)):
        assert list(nbr[at(*ijk)]) == [-1] * 6
    assert len(c0) + len(c1) == fitted.sum()
    for v in c0:
        a, r = divmod(int(flat[v]), 6)
        assert (a + r // 2 + r % 2) % 2 == 0
    for c in (c0, c1):
        assert np.all(np.diff(c) > 0) and fitted[c].all()
        assert not np.isin(nbr[c][nbr[c] >= 0], c).any()                         # no neighbour shares a colour
    # symmetric: q is a neighbour of v exactly when v is a neighbour of q (opposite face)
    for v in range(len(flat)):
        for k in range(6):
            q = nbr[v, k]
            if q >= 0:
                assert nbr[q, k ^ 1] == v


def _problem(V, n=24, m=20, seed=0):
    rng = np.random.default_rng(seed)
    T2 = np.logspace(1, np.log10(2000.0), n)
    t = 10.0 * np.arange(1, m + 1)
    D = np.exp(-t[:, None] / T2[None, :])
    truth = rng.uniform(0, 1, (V, n)) * (rng.random((V, n)) < 0.3)
    Y = truth @ D.T
    Y = Y / Y[:, :1] + rng.normal(0, 0.01, Y.shape)
    return D, Y


def test_mu_zero_is_the_point_problem():
    D, Y = _problem(6)
    L = 2.0 * np.eye(D.shape[1]) - np.eye(D.shape[1], k=1) - np.eye(D.shape[1], k=-1)
    for v, lam in enumerate((0.0, 1e-3, 0.05, 0.3, 1.8, 7.0)):
        x, mode = S.block_update(D, Y[v], L, lam, 0.0, np.full(D.shape[1], 5.0), 4)
        ref = O.nnls_tik(D, Y[v], L, lam)
        assert mode == 1 and np.array_equal(x > 0, ref > 0)
        assert np.abs(x - ref).max() <= 1e-10 * np.abs(ref).max()


def _volume(seed=3):
    rng = np.random.default_rng(seed)
    shape = (4, 3, 3)
    mask = rng.random(shape) < 0.8
    flat = np.nonzero(mask.ravel())[0]
    fitted = rng.random(len(flat)) < 0.9
    D, Y = _problem(len(flat), seed=seed)
    lam = rng.uniform(0.01, 0.5, len(flat))
    L = np.eye(D.shape[1])
    x0 = np.array([O.nnls_tik(D, Y[v], L, lam[v]) for v in range(len(flat))])
    return shape, flat, fitted, D, Y, lam, L, x0


def test_objective_does_not_increase_over_half_sweeps():
    shape, flat, fitted, D, Y, lam, L, x0 = _volume()
    nbr, colours = S.neighbours(flat, shape, fitted)
    mu = 0.2
    Dv = lambda v: D
    J = [S.objective(x0, fitted, Y, Dv, lam, L, nbr, mu)]
    _, trace = S.sweeps(x0, colours, Y, Dv, lam, L, nbr, mu, 3)
    J += [S.objective(x, fitted, Y, Dv, lam, L, nbr, mu) for x in trace]
    assert all(b <= a * (1 + 1e-12) for a, b in zip(J, J[1:])), J
    assert J[-1] < J[0]
    x = trace[-1]
    assert np.array_equal(x[~fitted], x0[~fitted])                     # voxels outside the fitted set stay


def test_result_does_not_depend_on_voxel_order():
    shape, flat, fitted, D, Y, lam, L, x0 = _volume(seed=4)
    nbr, colours = S.neighbours(flat, shape, fitted)
    Dv = lambda v: D
    x, _ = S.sweeps(x0, colours, Y, Dv, lam, L, nbr, 0.5, 2)
    rng = np.random.default_rng(0)
    perm = rng.permutation(len(flat))                                  # the masked-voxel list in another order
    inv = np.argsort(perm)
    nbr_p, col_p = S.neighbours(flat[perm], shape, fitted[perm])
    xp, _ = S.sweeps(x0[perm], col_p, Y[perm], Dv, lam[perm], L, nbr_p, 0.5, 2)
    assert np.array_equal(xp[inv] > 0, x > 0)
    assert np.abs(xp[inv] - x).max() <= 1e-12 * np.abs(x).max()
