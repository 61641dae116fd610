"""NumPy restatement of met2_mppca (csrc/met2_mppca.cu, whose header holds the definition), operation for operation:
the same IEEE +, -, *, / and sqrt in the same order, vectorised across voxels (elementwise IEEE operations do not
depend on the batch).  A voxel whose Jacobi iteration has stopped is a fixed point of further sweeps (every pair is
skipped: c = 1, s = t = 0), so the whole batch simply runs until its last voxel stops."""
import numpy as np

TINY = 2.0 ** -53
MAX_SWEEPS = 32


def window_starts(n, c, r):
    """Start s_a and length w_a of the window of centre coordinates c on an axis of size n."""
    w = min(2 * r + 1, n)
    return np.minimum(np.maximum(c - r, 0), n - w), w


def _rot(c, s, own_p, u, w):
    return np.where(own_p, c * u - s * w, s * w + c * u)


def jacobi(C):
    """Cyclic round-robin Jacobi of the kernel on C [B, N, N] -> (diag [B, N], V [B, N, N], sweeps [B] run per voxel,
    capped [B]: the voxel was still rotating after MAX_SWEEPS sweeps)."""
    B, N, _ = C.shape
    Np = N + (N & 1)
    m = Np - 1
    A = np.zeros((B, Np, Np))
    A[:, :N, :N] = C
    V = np.zeros((B, Np, Np))
    V[:, np.arange(N), np.arange(N)] = 1.0
    tr = np.zeros(B)
    for e in range(N):
        tr = tr + C[:, e, e]
    thr = TINY * tr
    idx = np.arange(Np)
    rows = np.arange(N)
    sweeps = np.zeros(B, dtype=np.int64)
    done = np.zeros(B, dtype=bool)
    for sweep in range(MAX_SWEEPS):
        any_rot = np.zeros(B, dtype=bool)
        for rr in range(m):
            mate = (2 * rr - idx) % m
            mate[rr] = m
            mate[m] = rr
            p, q = np.minimum(idx, mate), np.maximum(idx, mate)
            app, aqq, apq = A[:, p, p], A[:, q, q], A[:, p, q]             # [B, Np], per index
            rot = (q < N)[None, :] & ~(np.abs(apq) <= thr[:, None])
            with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
                theta = (aqq - app) / (2.0 * np.where(rot, apq, 1.0))
                t = 1.0 / (np.abs(theta) + np.sqrt(theta * theta + 1.0))
                t = np.where(theta < 0.0, -t, t)
                c = 1.0 / np.sqrt(t * t + 1.0)
                s = t * c
            c, s, t = np.where(rot, c, 1.0), np.where(rot, s, 0.0), np.where(rot, t, 0.0)
            any_rot |= rot.any(axis=1)
            # entry (i, j) of the new matrix, i, j < N
            mt = mate[:N]
            I, J = rows[:, None], rows[None, :]
            i2, j2 = mt[:, None], mt[None, :]
            ip, jp = I < i2, J < j2
            ci, si, cj, sj = c[:, :N, None], s[:, :N, None], c[:, None, :N], s[:, None, :N]
            x = A[:, :N, :N]
            x_j2 = A[:, :N][:, :, mt]
            x_i2 = A[:, mt][:, :, :N]
            x_i2j2 = A[:, mt][:, :, mt]
            first = np.minimum(I, i2) < np.minimum(J, j2)
            a = _rot(ci, si, ip, _rot(cj, sj, jp, x, x_j2), _rot(cj, sj, jp, x_i2, x_i2j2))
            b = _rot(cj, sj, jp, _rot(ci, si, ip, x, x_i2), _rot(ci, si, ip, x_j2, x_i2j2))
            new = np.where(first, a, b)
            same = (J == I) | (J == i2)
            tI, appI, aqqI, apqI, rotI = t[:, :N, None], app[:, :N, None], aqq[:, :N, None], apq[:, :N, None], rot[:, :N, None]
            diag_p = appI - tI * apqI
            diag_q = aqqI + tI * apqI
            offd = np.where(rotI, 0.0, apqI)
            blk = np.where(J == I, np.where(ip, diag_p, diag_q), offd)
            new = np.where(same, blk, new)
            Vn = _rot(cj, sj, jp, V[:, :N, :N], V[:, :N][:, :, mt])
            A[:, :N, :N] = new
            V[:, :N, :N] = Vn
        sweeps += ~done
        done |= ~any_rot
        if done.all():
            break
    return np.diagonal(A[:, :N, :N], axis1=1, axis2=2).copy(), V[:, :N, :N].copy(), sweeps, ~done


def mp_classify(ev, N, M):
    """Step 5 on ascending eigenvalues ev [B, N] -> (sigma^2 [B], n_noise [B])."""
    R, Q = min(N, M - 1), float(max(N, M - 1))
    off = N - R
    lam = np.where(ev > 0.0, ev, 0.0) / Q
    S = np.zeros(ev.shape[0])
    sigma2 = np.zeros(ev.shape[0])
    cut = np.zeros(ev.shape[0], dtype=np.int64)
    l0 = lam[:, off]
    for p in range(R):
        lp = lam[:, off + p]
        S = S + lp
        gamma = float(p + 1) / Q
        s1 = S / float(p + 1)
        s2 = (lp - l0) / (4.0 * np.sqrt(gamma))
        hit = s2 < s1
        sigma2 = np.where(hit, s1, sigma2)
        cut = np.where(hit, p + 1, cut)
    return sigma2, cut + off


def _windows(vol, centres, r):
    """Samples X [B, M, N] of the windows of the voxels `centres` [B, 3], in C order."""
    nx, ny, nz, N = vol.shape
    sx, wx = window_starts(nx, centres[:, 0], r)
    sy, wy = window_starts(ny, centres[:, 1], r)
    sz, wz = window_starts(nz, centres[:, 2], r)
    di, dj, dk = np.meshgrid(np.arange(wx), np.arange(wy), np.arange(wz), indexing="ij")
    di, dj, dk = di.ravel(), dj.ravel(), dk.ravel()
    return vol[sx[:, None] + di, sy[:, None] + dj, sz[:, None] + dk], wx * wy * wz


def mppca_batch(vol, centres, r, eig=None):
    """Outputs of the voxels `centres` [B, 3] -> dict(out [B, N], sigma [B], n_signal [B], plus the intermediates).
    eig: None for the kernel's Jacobi, or a function C -> (ascending eigenvalues, eigenvectors as columns)."""
    N = vol.shape[3]
    X, M = _windows(vol, centres, r)
    B = X.shape[0]
    bad = ~np.isfinite(X).all(axis=(1, 2))
    X = np.where(bad[:, None, None], 0.0, X)
    acc = np.zeros((B, N))
    for s in range(M):
        acc = acc + X[:, s]
    mu = acc / float(M)
    C = np.zeros((B, N, N))
    for s in range(M):
        xc = X[:, s] - mu
        C = C + xc[:, :, None] * xc[:, None, :]
    info = {}
    if eig is None:
        d, V, sweeps, capped = jacobi(C)
        order = np.argsort(d, axis=1, kind="stable")          # ascending, ties: lower index
        ev = np.take_along_axis(d, order, axis=1)
        W = np.take_along_axis(V, order[:, None, :], axis=2)
        info.update(sweeps=sweeps, capped=capped)
    else:
        ev, W = eig(C)
    sigma2, n_noise = mp_classify(ev, N, M)
    xcen = vol[centres[:, 0], centres[:, 1], centres[:, 2]]
    d = np.where(bad[:, None], 0.0, xcen) - mu
    sig_comp = np.arange(N)[None, :] >= n_noise[:, None]                 # [B, pos]
    t = np.zeros((B, N))
    for e in range(N):
        t = t + W[:, e, :] * d[:, e:e + 1]
    t = np.where(sig_comp, t, 0.0)
    acc = np.zeros((B, N))
    for pos in range(N):
        acc = np.where(sig_comp[:, pos:pos + 1], acc + W[:, :, pos] * t[:, pos:pos + 1], acc)
    x = mu + acc
    out = np.where(x > 0.0, x, 0.0)
    out = np.where(bad[:, None], xcen, out)
    sigma = np.where(bad, np.nan, np.sqrt(sigma2))
    n_signal = np.where(bad, -1, N - n_noise).astype(np.int32)
    info.update(out=out, sigma=sigma, n_signal=n_signal, ev=ev, M=M, n_noise=n_noise)
    return info


def mppca(vol, mask, r=2, eig=None, batch=512, info=False):
    """met2_mppca on host arrays: vol [nx, ny, nz, N], mask [nx, ny, nz] -> (out like vol, sigma [nx, ny, nz],
    n_signal [nx, ny, nz] int32), plus the per-voxel sweep counts / cap flags and eigenvalues of the kernel's Jacobi
    when info=True."""
    vol = np.ascontiguousarray(vol, dtype=np.float64)
    shape = vol.shape[:3]
    out = np.zeros_like(vol)
    sigma = np.zeros(shape)
    n_signal = np.zeros(shape, dtype=np.int32)
    centres = np.argwhere(np.asarray(mask) == 1)
    extra = dict(sweeps=[], capped=[], ev=[], centres=centres)
    for lo in range(0, len(centres), batch):
        c = centres[lo:lo + batch]
        res = mppca_batch(vol, c, r, eig)
        out[c[:, 0], c[:, 1], c[:, 2]] = res["out"]
        sigma[c[:, 0], c[:, 1], c[:, 2]] = res["sigma"]
        n_signal[c[:, 0], c[:, 1], c[:, 2]] = res["n_signal"]
        for k in ("sweeps", "capped", "ev"):
            if k in res:
                extra[k].append(res[k])
    if info:
        for k in ("sweeps", "capped", "ev"):
            extra[k] = np.concatenate(extra[k]) if extra[k] else np.zeros(0)
        return out, sigma, n_signal, extra
    return out, sigma, n_signal
