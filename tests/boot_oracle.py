"""NumPy restatement of the per-voxel bootstrap of csrc/met2_boot.cu (the definition is in that file's header comment):
wild-bootstrap replicates with Rademacher signs drawn from SplitMix64, and the per-voxel summary of the refitted maps
(mean, sd, 2.5th / 97.5th percentile over the valid replicates).  Used by the emulator and GPU tests as the reference
the kernels must equal bit for bit."""
import numpy as np

GOLDEN = np.uint64(0x9E3779B97F4A7C15)
MIX1 = np.uint64(0xBF58476D1CE4E5B9)
MIX2 = np.uint64(0x94D049BB133111EB)
ST_SKIPPED = 1
QUANTILES = (2.5, 97.5)


def splitmix64(seed, k):
    """h = splitmix64(seed, k) for an array of counters k (uint64 arithmetic, mod 2^64)."""
    k = np.asarray(k, dtype=np.uint64)
    with np.errstate(over="ignore"):
        x = np.uint64(seed) + (k + np.uint64(1)) * GOLDEN
        x = (x ^ (x >> np.uint64(30))) * MIX1
        x = (x ^ (x >> np.uint64(27))) * MIX2
    return x ^ (x >> np.uint64(31))


def signs(V, B, nTE, seed=0, voxel_offset=0):
    """bool [V, B, nTE]: True where bit e of h(g * B + b) is set, i.e. where the residual is subtracted."""
    g = np.arange(V, dtype=np.uint64) + np.uint64(voxel_offset)
    k = g[:, None] * np.uint64(B) + np.arange(B, dtype=np.uint64)[None, :]
    h = splitmix64(seed, k)
    bits = (h[:, :, None] >> np.arange(nTE, dtype=np.uint64)[None, None, :]) & np.uint64(1)
    return bits.astype(bool)


def resample(sig, est_signal, fa_index, B, seed=0, voxel_offset=0):
    """-> rep_sig [V * B, nTE], rep_fa_index [V * B] (rows r = v * B + b)."""
    sig = np.asarray(sig, dtype=np.float64)
    est = np.asarray(est_signal, dtype=np.float64)
    V, nTE = sig.shape
    r = sig - est
    neg = signs(V, B, nTE, seed, voxel_offset)
    rep = np.where(neg, (est - r)[:, None, :], (est + r)[:, None, :])
    rep_fa = np.repeat(np.asarray(fa_index, dtype=np.int32), B)
    return rep.reshape(V * B, nTE), rep_fa


def summarise_values(x):
    """(mean, sd, p2.5, p97.5) of the valid values x of one voxel and map, in replicate order."""
    n = len(x)
    if n == 0:
        return (0.0, 0.0, 0.0, 0.0)
    if np.isnan(x).any():
        return (np.nan,) * 4
    s = 0.0
    for v in x:           # sequential, in replicate order
        s = s + v
    mean = s / n
    sd = 0.0
    if n > 1:
        ss = 0.0
        for v in x:
            d = v - mean
            ss = ss + d * d
        sd = float(np.sqrt(ss / (n - 1)))
    p = np.percentile(np.asarray(x, dtype=np.float64), QUANTILES, method="linear")
    return (float(mean), sd, float(p[0]), float(p[1]))


def summary(rep_maps, rep_status, B):
    """rep_maps [V * B, 6], rep_status [V * B] -> (stats [V, 6, 4], n_valid [V] int32)."""
    rep_maps = np.asarray(rep_maps, dtype=np.float64).reshape(-1, B, 6)
    valid = (np.asarray(rep_status).astype(np.uint32).reshape(-1, B) & ST_SKIPPED) == 0
    V = rep_maps.shape[0]
    stats = np.zeros((V, 6, 4))
    for v in range(V):
        vals = rep_maps[v][valid[v]]
        for m in range(6):
            stats[v, m] = summarise_values(vals[:, m])
    return stats, valid.sum(axis=1).astype(np.int32)
