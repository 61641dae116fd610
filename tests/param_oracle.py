"""NumPy restatement of the three-pool parametric T2 fit of csrc/met2_param.cu (met2_param_fit), line for line with the
definition in that file's header: the EPG recurrence of met2_epg.cuh with forward-mode derivatives, the start from the
point fit's spectrum, and the projected Levenberg-Marquardt iteration.  The voxels run in lockstep, each with its own
state; the arithmetic of each voxel is the kernel's.  The kernel's sums over echoes are butterfly sums, here np.einsum,
so results agree to rounding, not bit for bit."""
import numpy as np

ST_SKIPPED, ST_NONFINITE, ST_ITMAX, ST_AT_BOUND = 1, 2, 4, 64
DEFAULTS = dict(mu0=1e-3, mu_max=1e16, ftol=1e-12, xtol=1e-10, max_iter=2000)


class Dual:
    """value, d/du (u = ln T2) and d/dalpha (deg); the operations of met2::Dual."""
    __slots__ = ("v", "t", "a")

    def __init__(self, v, t, a):
        self.v, self.t, self.a = v, t, a

    def __add__(x, y):
        return Dual(x.v + y.v, x.t + y.t, x.a + y.a)

    def __sub__(x, y):
        return Dual(x.v - y.v, x.t - y.t, x.a - y.a)

    def __mul__(x, y):
        if isinstance(y, Dual):
            return Dual(x.v * y.v, x.t * y.v + x.v * y.t, x.a * y.v + x.v * y.a)
        return Dual(x.v * y, x.t * y, x.a * y)

    def __rmul__(x, s):
        return Dual(s * x.v, s * x.t, s * x.a)

    def __truediv__(x, s):
        return Dual(x.v / s, x.t / s, x.a / s)

    def __rtruediv__(x, s):
        r = s / x.v
        d = -r / x.v
        return Dual(r, d * x.t, d * x.a)

    def map(self, f):
        return Dual(f(self.v), f(self.t), f(self.a))


def dexp(x):
    e = np.exp(x.v)
    return Dual(e, e * x.t, e * x.a)


def dsin(x):
    s, c = np.sin(x.v), np.cos(x.v)
    return Dual(s, c * x.t, c * x.a)


def dcos(x):
    s, c = np.sin(x.v), np.cos(x.v)
    return Dual(c, -s * x.t, -s * x.a)


def epg_curves(alpha, T2, T1, tau, TR, n):
    """d(T2, alpha) of met2_param.cu (the met2_epg_dictionary column) with d/du and d/dalpha, for arrays alpha (deg) and
    T2 (ms) of one shape S.  Returns three arrays [*S, n]."""
    alpha = np.asarray(alpha, dtype=np.float64)[..., None]
    T2 = np.asarray(T2, dtype=np.float64)[..., None]
    shape = np.broadcast(alpha, T2).shape
    zero = np.zeros(shape)
    al = Dual(alpha + zero, zero, zero + 1.0)
    t2 = Dual(T2 + zero, T2 + zero, zero)
    # epg_coef
    rad = 3.14159265358979323846 / 180.0
    a = al * rad
    a_exc = (al / 2.0) * rad
    half = tau / 2.0
    e2 = dexp(-half * (1.0 / t2))
    e1 = np.exp(-half * (1.0 / T1))
    ch, sh = dcos(a / 2.0), dsin(a / 2.0)
    c2, s2, sa, ca = ch * ch, sh * sh, dsin(a), dcos(a)
    F0 = dsin(a_exc)
    state = np.zeros(shape[:-1] + (n + 1,))
    Fp, Fm, Z = (Dual(state.copy(), state.copy(), state.copy()) for _ in range(3))
    fm1 = dcos(a_exc)
    for part in ("v", "t", "a"):
        getattr(Fm, part)[..., 1] = getattr(fm1, part)[..., 0]
    scale = 1.0 - np.exp(-TR / T1)
    out = Dual(np.zeros(shape[:-1] + (n,)), np.zeros(shape[:-1] + (n,)), np.zeros(shape[:-1] + (n,)))
    for echo in range(n):
        for half_step in range(2):
            # shift: F0 <- F-1, F+k <- F+(k-1), F+1 <- F0, F-k <- F-(k+1), F-n <- 0
            newF0 = Fm.map(lambda x: x[..., 1:2].copy())
            for part in ("v", "t", "a"):
                fp, fm = getattr(Fp, part), getattr(Fm, part)
                fp[..., 2:n + 1] = fp[..., 1:n].copy()
                fp[..., 1] = getattr(F0, part)[..., 0]
                fm[..., 1:n] = fm[..., 2:n + 1].copy()
                fm[..., n] = 0.0
            F0 = newF0 * e2
            # relaxation (epg_relax)
            Fp, Fm, Z = Fp * e2, Fm * e2, Z * e1
            if half_step == 0:   # RF mixing (epg_rf)
                p, m, q = Fp, Fm, Z
                Fp = c2 * p + s2 * m + sa * q
                Fm = s2 * p + c2 * m - sa * q
                Z = (-0.5 * sa) * p + (0.5 * sa) * m + ca * q
        o = scale * F0
        out.v[..., echo], out.t[..., echo], out.a[..., echo] = o.v[..., 0], o.t[..., 0], o.a[..., 0]
    return out.v, out.t, out.a


def evaluate(p, y, T1, tau, TR):
    """m [N, n], F [N], g [N, 7], H [N, 7, 7] at p [N, 7] for y [N, n]."""
    n = y.shape[1]
    d, dt, da = epg_curves(np.repeat(p[:, 6:7], 3, axis=1), np.exp(p[:, 3:6]), T1, tau, TR, n)
    A = p[:, 0:3, None]
    m = A[:, 0] * d[:, 0] + A[:, 1] * d[:, 1] + A[:, 2] * d[:, 2]
    J = np.stack([d[:, 0], d[:, 1], d[:, 2], A[:, 0] * dt[:, 0], A[:, 1] * dt[:, 1], A[:, 2] * dt[:, 2],
                  A[:, 0] * da[:, 0] + A[:, 1] * da[:, 1] + A[:, 2] * da[:, 2]], axis=-1)
    r = m - y
    F = 0.5 * np.einsum("ne,ne->n", r, r)
    g = np.einsum("nei,ne->ni", J, r)
    H = np.einsum("nei,nej->nij", J, J)
    return m, F, g, H, J


def box(cfg):
    lo = np.array([0.0, 0.0, 0.0] + list(np.log(cfg["t2_lo"])) + [cfg["fa_lo"]])
    hi = np.array([np.inf] * 3 + list(np.log(cfg["t2_hi"])) + [cfg["fa_hi"]])
    return lo, hi


def start(x, logT2, comp, fa_deg, lo, hi):
    """p0 [N, 7] from the normalised spectra x [N, nT2] and the FA stage's angles."""
    p = np.zeros((x.shape[0], 7))
    for c in range(3):
        sel = (comp & (1 << c)) != 0
        a = x[:, sel].sum(axis=1)
        w = (x[:, sel] * logT2[sel]).sum(axis=1)
        p[:, c] = a
        with np.errstate(invalid="ignore", divide="ignore"):
            u = np.where(a > 0.0, w / np.where(a > 0.0, a, 1.0), 0.5 * (lo[3 + c] + hi[3 + c]))
        p[:, 3 + c] = np.minimum(np.maximum(u, lo[3 + c]), hi[3 + c])
    p[:, 6] = np.minimum(np.maximum(fa_deg, lo[6]), hi[6])
    return p


def _solve(H, g, fr, mu):
    """delta of step 3 for one voxel, or None when a pivot is not positive."""
    L = np.zeros((7, 7))
    for i in range(7):
        for j in range(i + 1):
            if i == j:
                mij = H[i, i] + mu * H[i, i] if fr[i] else 1.0
            else:
                mij = H[i, j] if fr[i] and fr[j] else 0.0
            for k in range(j):
                mij -= L[i, k] * L[j, k]
            if i == j:
                if not mij > 0.0:
                    return None
                L[i, i] = np.sqrt(mij)
            else:
                L[i, j] = mij / L[j, j]
    b = np.zeros(7)
    for i in range(7):
        s = -g[i] if fr[i] else 0.0
        for k in range(i):
            s -= L[i, k] * b[k]
        b[i] = s / L[i, i]
    for i in range(6, -1, -1):
        s = b[i]
        for k in range(i + 1, 7):
            s -= L[k, i] * b[k]
        b[i] = s / L[i, i]
    return b


def param_fit(sig, fa_deg, fsol, status, logT2, comp, cfg):
    """met2_param_fit.  cfg: dict(tau, TR, T1, t2_lo[3], t2_hi[3], fa_lo, fa_hi) and optionally the DEFAULTS keys.
    Returns dict(params, maps, est_signal, sse, iters, status) like the kernel."""
    cfg = {**DEFAULTS, **cfg}
    sig = np.asarray(sig, dtype=np.float64)
    V, nTE = sig.shape
    status = np.asarray(status).astype(np.uint32)
    comp = np.asarray(comp, dtype=np.uint8)
    logT2 = np.asarray(logT2, dtype=np.float64)
    out = dict(params=np.zeros((V, 7)), maps=np.zeros((V, 6)), est_signal=np.zeros((V, nTE)), sse=np.zeros(V),
               iters=np.zeros(V, dtype=np.int32), status=(status & (ST_SKIPPED | ST_NONFINITE)).astype(np.uint32))
    idx = np.nonzero(out["status"] == 0)[0]
    if len(idx) == 0:
        return out
    T1, tau, TR = cfg["T1"], cfg["tau"], cfg["TR"]
    lo, hi = box(cfg)
    s0 = sig[idx, 0]
    y = sig[idx] / s0[:, None]
    p = start(np.asarray(fsol, dtype=np.float64)[idx] / s0[:, None], logT2, comp,
              np.asarray(fa_deg, dtype=np.float64)[idx], lo, hi)
    m, F, g, H, _ = evaluate(p, y, T1, tau, TR)
    N = len(idx)
    mu = np.full(N, float(cfg["mu0"]))
    it = np.zeros(N, dtype=np.int32)
    st = np.zeros(N, dtype=np.uint32)
    active = np.ones(N, dtype=bool)
    while active.any():
        trial = []
        for v in np.nonzero(active)[0]:
            if it[v] == cfg["max_iter"]:                                           # 1
                st[v] |= ST_ITMAX
                active[v] = False
                continue
            it[v] += 1
            fr = ~((np.diag(H[v]) == 0.0) | ((p[v] <= lo) & (g[v] > 0.0)) | ((p[v] >= hi) & (g[v] < 0.0)))   # 2
            if not fr.any():
                active[v] = False
                continue
            b = _solve(H[v], g[v], fr, mu[v])                                      # 3
            if b is None:
                mu[v] *= 10.0
                if mu[v] > cfg["mu_max"]:
                    active[v] = False
                continue
            t = np.where(fr, np.minimum(np.maximum(p[v] + b, lo), hi), p[v])       # 4
            dn = pn = 0.0
            for i in range(7):
                dn += (t[i] - p[v, i]) * (t[i] - p[v, i])
                pn += p[v, i] * p[v, i]
            if np.sqrt(dn) <= cfg["xtol"] * (cfg["xtol"] + np.sqrt(pn)):
                active[v] = False
                continue
            trial.append((v, t))
        if not trial:
            continue
        tv = np.array([v for v, _ in trial])
        tp = np.array([t for _, t in trial])
        mt, Ft, gt, Ht, _ = evaluate(tp, y[tv], T1, tau, TR)                       # 5
        for k, v in enumerate(tv):
            if Ft[k] < F[v]:
                done = F[v] - Ft[k] <= cfg["ftol"] * F[v]
                p[v], g[v], H[v], m[v], F[v] = tp[k], gt[k], Ht[k], mt[k], Ft[k]
                mu[v] /= 10.0
                if done:
                    active[v] = False
            else:
                mu[v] *= 10.0
                if mu[v] > cfg["mu_max"]:
                    active[v] = False
    at = np.any((p[:, 3:] == lo[3:]) | (p[:, 3:] == hi[3:]), axis=1)
    st |= np.where(at, ST_AT_BOUND, 0).astype(np.uint32)
    sumA = p[:, 0] + p[:, 1] + p[:, 2]
    params = np.concatenate([p[:, :3] * s0[:, None], np.exp(p[:, 3:6]), p[:, 6:7]], axis=1)
    with np.errstate(invalid="ignore", divide="ignore"):
        fr = np.where(sumA[:, None] > 0.0, p[:, :3] / np.where(sumA > 0.0, sumA, 1.0)[:, None], 0.0)
    maps = np.stack([fr[:, 0], fr[:, 1], fr[:, 2], np.where(p[:, 0] > 0.0, params[:, 3], 0.0),
                     np.where(p[:, 1] > 0.0, params[:, 4], 0.0), s0 * sumA], axis=1)
    out["params"][idx] = params
    out["maps"][idx] = maps
    out["est_signal"][idx] = s0[:, None] * m
    out["sse"][idx] = (s0 * s0) * (2.0 * F)
    out["iters"][idx] = it
    out["status"][idx] = st
    return out


def plan_cfg(T2s, myelin_T2=40.0, tau=10.0, TR=1000.0, T1=1000.0, **kw):
    """The box batched.Met2Plan.param_fit builds: T2s[0] / myelin_T2 / 200 / T2s[-1], flip angle 90-180."""
    return dict(tau=tau, TR=TR, T1=T1, t2_lo=[T2s[0], myelin_T2, 200.0], t2_hi=[myelin_T2, 200.0, T2s[-1]],
                fa_lo=90.0, fa_hi=180.0, **kw)
