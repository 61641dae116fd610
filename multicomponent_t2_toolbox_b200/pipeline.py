"""Volume-level driver: what motor_recon_met2 does between "arrays are in host memory" and "arrays are handed to the
NIfTI writer" (motor/motor_recon_met2_real_data.py:167-182, 279, 349-373, 428-472), as gather -> two batched GPU calls
-> scatter.  Also holds the voxel-slab partition used for multi-GPU runs (SURVEY.md §8e): voxels are independent, so
each rank fits a contiguous slab of the masked-voxel list and no collective runs during the fit.
"""
import os
import time

import numpy as np
import torch

from . import batched

MAP_NAMES = ("MWF", "IEWF", "FWF", "T2_M", "T2_IE", "TWC")


def slab_bounds(n_voxels, rank, world_size):
    """Contiguous slab [lo, hi) of rank `rank` out of `world_size`: ceil(V / W) voxels per rank, last ranks may be short
    or empty.  Every voxel belongs to exactly one rank; concatenating the slabs in rank order restores the list."""
    if world_size < 1 or not (0 <= rank < world_size):
        raise ValueError("bad rank/world_size")
    per = -(-int(n_voxels) // int(world_size)) if n_voxels > 0 else 0
    lo = min(n_voxels, rank * per)
    hi = min(n_voxels, lo + per)
    return lo, hi


def cyclic_slab(n_voxels, rank, world_size, chunk=2048):
    """Block-cyclic alternative to `slab_bounds` (SURVEY.md §8e: over-decomposition for load balance — the cost of a
    voxel depends on its flip angle and spectrum, and both vary smoothly across the volume): chunks of `chunk`
    consecutive voxels are dealt to the ranks round-robin.  Returns this rank's voxel indices (sorted, int64); the
    ranks' index sets are disjoint and cover [0, n_voxels)."""
    if world_size < 1 or not (0 <= rank < world_size) or chunk < 1:
        raise ValueError("bad rank/world_size/chunk")
    idx = np.arange(int(n_voxels), dtype=np.int64)
    return idx[(idx // int(chunk)) % int(world_size) == rank]


def masked_voxel_list(data, mask, premasked=False):
    """Return (flat voxel indices, signals[V,nTE]) of the voxels with mask > 0, in C order of (x, y, z).  Unless
    `premasked` (the motor entry points have already done it, motor...:178-180,279 — applying a label mask twice would
    scale the data by mask squared), the mask multiplication and the negative clamp are applied here."""
    nx, ny, nz, nt = data.shape
    m = np.asarray(mask).reshape(-1)
    flat = np.nonzero(m > 0)[0]
    sig = np.ascontiguousarray(data.reshape(-1, nt)[flat], dtype=np.float64)
    if not premasked:
        sig = sig * m[flat][:, None]
        sig[sig < 0.0] = 0.0
    return flat, sig


def chunk_deal(n_voxels, n_parts, chunks_per_part=4, align=64):
    """Over-decomposed contiguous partition for ONE volume spread over `n_parts` GPUs: the voxel list is cut into
    ~n_parts * chunks_per_part contiguous chunks (multiples of `align` voxels) that are dealt round-robin, so that
    every part gets voxels from all over the volume (per-voxel cost follows the flip angle and the spectrum, which vary
    smoothly in space) while host <-> device traffic stays a handful of large contiguous copies per part.
    Returns a list (one entry per part) of lists of (lo, hi); the ranges are disjoint and cover [0, n_voxels)."""
    if n_parts < 1 or chunks_per_part < 1:
        raise ValueError("bad n_parts/chunks_per_part")
    n_voxels = int(n_voxels)
    nchunks = n_parts * chunks_per_part
    size = -(-n_voxels // nchunks) if n_voxels > 0 else 0
    size = max(align, -(-size // align) * align)
    parts = [[] for _ in range(n_parts)]
    k, lo = 0, 0
    while lo < n_voxels:
        hi = min(n_voxels, lo + size)
        parts[k % n_parts].append((lo, hi))
        lo = hi
        k += 1
    return parts


def spatial_neighbours(flat, shape, fitted):
    """Neighbour table and red-black colours of the spatially regularised fit (`batched.Met2Plan.spatial_fit`).
    flat[V]: C-order indices of the masked voxels in a volume of `shape` (nx, ny, nz), as `masked_voxel_list` returns
    them; fitted[V]: the voxels the point fit did not skip.  Returns nbr int32 [V, 6] (positions in 0..V-1 of the
    fitted face neighbours in the order -x, +x, -y, +y, -z, +z; -1 = none, and all -1 for a voxel that is not fitted)
    and the two colour lists (positions of the fitted voxels with (i + j + k) % 2 == 0 and == 1, ascending)."""
    nx, ny, nz = (int(s) for s in shape)
    flat = np.asarray(flat, dtype=np.int64)
    fitted = np.asarray(fitted, dtype=bool)
    where = np.full(nx * ny * nz, -1, dtype=np.int64)
    where[flat[fitted]] = np.nonzero(fitted)[0]
    i, j, k = np.unravel_index(flat, (nx, ny, nz))
    nbr = np.full((len(flat), 6), -1, dtype=np.int32)
    for f, (di, dj, dk) in enumerate(((-1, 0, 0), (1, 0, 0), (0, -1, 0), (0, 1, 0), (0, 0, -1), (0, 0, 1))):
        a, b, c = i + di, j + dj, k + dk
        inside = fitted & (a >= 0) & (a < nx) & (b >= 0) & (b < ny) & (c >= 0) & (c < nz)
        nbr[inside, f] = where[(a[inside] * ny + b[inside]) * nz + c[inside]]
    colour = (i + j + k) % 2
    colours = tuple(np.nonzero(fitted & (colour == c))[0].astype(np.int32) for c in (0, 1))
    return nbr, colours


# The per-voxel outputs of the stages: name, trailing shape (ints and Met2Plan attributes), dtype, and the stage that
# produces it.  "fa" always runs, "t2" unless fa_only, "bootstrap" when n_bootstrap > 0, "parametric" when parametric,
# "rician" when a noise sigma is given.
VOXEL_OUTPUTS = (
    ("fa_index", (), torch.int32, "fa"), ("fa_deg", (), torch.float64, "fa"), ("km", (), torch.float64, "fa"),
    ("fa_status", (), torch.int32, "fa"),
    ("fsol", ("npc",), torch.float64, "t2"), ("est_signal", ("nTE",), torch.float64, "t2"),
    ("reg", (), torch.float64, "t2"), ("maps", (6,), torch.float64, "t2"), ("status", (), torch.int32, "t2"),
    ("boot_stats", (6, 4), torch.float64, "bootstrap"), ("boot_n_valid", (), torch.int32, "bootstrap"),
    ("param_params", (7,), torch.float64, "parametric"), ("param_maps", (6,), torch.float64, "parametric"),
    ("param_est_signal", ("nTE",), torch.float64, "parametric"), ("param_sse", (), torch.float64, "parametric"),
    ("param_iters", (), torch.int32, "parametric"), ("param_status", (), torch.int32, "parametric"),
    ("rician_fsol", ("npc",), torch.float64, "rician"), ("rician_est_signal", ("nTE",), torch.float64, "rician"),
    ("rician_maps", (6,), torch.float64, "rician"), ("rician_iters", (), torch.int32, "rician"),
    ("rician_status", (), torch.int32, "rician"))

# the volumes of the three-pool parametric fit: name -> (output, column)
PARAM_VOLUMES = {"MWF_3pool": ("param_maps", 0), "IEWF_3pool": ("param_maps", 1), "FWF_3pool": ("param_maps", 2),
                 "T2_M_3pool": ("param_maps", 3), "T2_IE_3pool": ("param_maps", 4), "T2_FW_3pool": ("param_params", 5),
                 "FA_3pool": ("param_params", 6), "TWC_3pool": ("param_maps", 5), "SSE_3pool": ("param_sse", None),
                 "Est_Signal_3pool": ("param_est_signal", None)}

# the volumes of the Rician-likelihood fit: name -> (output, column)
RICIAN_VOLUMES = {**{name + "_rician": ("rician_maps", i) for i, name in enumerate(MAP_NAMES)},
                  "fsol_4D_rician": ("rician_fsol", None), "Est_Signal_rician": ("rician_est_signal", None),
                  "rician_iters": ("rician_iters", None)}

# The volumes of `recon_arrays`: name, per-voxel output, column (None: all of it) and dtype.  A volume is returned when
# its per-voxel output was computed.
VOLUMES = (("FA", "fa_deg", None, np.float64), ("FA_index", "fa_index", None, np.float64),
           *((name, "maps", i, np.float64) for i, name in enumerate(MAP_NAMES)),
           ("reg_param", "reg", None, np.float64), ("fsol_4D", "fsol", None, np.float64),
           ("Est_Signal", "est_signal", None, np.float64), ("status", "status", None, np.int32),
           *((name + "_bootstrap", "boot_stats", i, np.float64) for i, name in enumerate(MAP_NAMES)),
           ("bootstrap_n_valid", "boot_n_valid", None, np.int32),
           *((name, key, col, np.float64) for name, (key, col) in PARAM_VOLUMES.items()),
           *((name, key, col, np.int32 if key == "rician_iters" else np.float64)
             for name, (key, col) in RICIAN_VOLUMES.items()))


def _fa_stage(plan, s):
    fa = s["fa"] = plan.fa_fit(s["sig_fa"], out=s["fa"])
    return dict(fa_index=fa["fa_index"], fa_deg=fa["fa_deg"], km=fa["km"], fa_status=fa["status"])


def _t2_stage(plan, s):
    s["t2"] = plan.t2_fit(s["sig"], s["fa"]["fa_index"], out=s["t2"])
    return dict(s["t2"])


def _bootstrap_stage(plan, s, n_bootstrap, seed):
    """`Met2Plan.bootstrap` from the point fit, one call per contiguous range of s["ranges"] with voxel_offset = the
    range's start in the whole voxel list (a voxel's replicates depend on that position).  Voxels the point fit skipped
    get zeros, like their maps."""
    t2, fa_index = s["t2"], s["fa"]["fa_index"]
    parts, o = [], 0
    for lo, hi in s["ranges"]:
        rows = slice(o, o + hi - lo)
        parts.append(plan.bootstrap(s["sig"][rows], fa_index[rows], t2["est_signal"][rows], B=n_bootstrap, seed=seed,
                                    voxel_offset=lo))
        o += hi - lo
    stats, n_valid = (torch.cat(p) for p in zip(*parts))
    skipped = (t2["status"] & batched.ST_SKIPPED) != 0
    stats.masked_fill_(skipped[:, None, None], 0.0)
    n_valid.masked_fill_(skipped, 0)
    return dict(boot_stats=stats, boot_n_valid=n_valid)


def _param_stage(plan, s):
    """`Met2Plan.param_fit` started from the point fit; T2_FW (params column 5) is zeroed where the free-water
    amplitude is 0, like T2_M and T2_IE in the maps."""
    pf = plan.param_fit(s["sig"], s["fa"]["fa_deg"], s["t2"]["fsol"], s["t2"]["status"])
    pf["params"][:, 5].masked_fill_(pf["params"][:, 2] <= 0.0, 0.0)
    return {"param_" + k: v for k, v in pf.items()}


def _rician_stage(plan, s):
    """`Met2Plan.rician_fit` started from the point fit, with lambda from a second `t2_fit` under REG_IS_LAMBDA (the
    point fit's reg is k_est for X2) and the per-voxel noise sigma s["sigma"]."""
    lam = plan.t2_fit(s["sig"], s["fa"]["fa_index"], flags=batched.REG_IS_LAMBDA)["reg"]
    rf = plan.rician_fit(s["sig"], s["fa"]["fa_index"], lam, s["sigma"], s["t2"]["fsol"], s["t2"]["status"])
    return {"rician_" + k: rf[k] for k in ("fsol", "est_signal", "maps", "iters", "status")}


def _stages(fa_only=False, n_bootstrap=0, bootstrap_seed=0, parametric=False, rician=False):
    """The per-voxel stages in order, as (name, stage).  A stage takes (plan, s), s: the device state of one set of
    voxels (sig, sig_fa, sigma for the Rician fit, ranges: their (lo, hi) in the whole voxel list, and the fa / t2
    results, reused as `out=`), and returns its VOXEL_OUTPUTS as CUDA tensors, enqueued on the current stream.
    Bootstrap, the parametric and the Rician fit start from the point fit."""
    stages = [("fa", _fa_stage)]
    if not fa_only:
        stages.append(("t2", _t2_stage))
        if n_bootstrap > 0:
            stages.append(("bootstrap", lambda plan, s: _bootstrap_stage(plan, s, n_bootstrap, bootstrap_seed)))
        if parametric:
            stages.append(("parametric", _param_stage))
        if rician:
            stages.append(("rician", _rician_stage))
    return stages


def _outputs(stages):
    """The entries of VOXEL_OUTPUTS that `stages` produce."""
    ran = {name for name, _ in stages}
    return [o for o in VOXEL_OUTPUTS if o[3] in ran]


def host_buffers(plan, V, pinned=True, n_bootstrap=0, parametric=False, rician=False):
    """Host (pinned) arrays for the outputs of `fit_voxels` / `MultiGpuFit.fit` of V voxels: the per-voxel outputs of
    the point fit, plus those of the bootstrap (n_bootstrap > 0), of the parametric fit and of the Rician fit, and
    fsol_sum[npc]."""
    pin = pinned and torch.cuda.is_available()
    bufs = {name: torch.empty((V,) + tuple(getattr(plan, n) if isinstance(n, str) else n for n in shape), dtype=dtype,
                              pin_memory=pin)
            for name, shape, dtype, _ in _outputs(_stages(n_bootstrap=n_bootstrap, parametric=parametric,
                                                            rician=rician))}
    bufs["fsol_sum"] = torch.empty(plan.npc, dtype=torch.float64, pin_memory=pin)
    return bufs


def _whole_volume(plan, sig, fa_index, fsol_sum, in_mask=None, roi=None, spatial=None, fsol=None, status=None):
    """The steps that need every voxel on one device (plan.dev), from sig[V, nTE] and fa_index[V] (CUDA): the
    mean-spectrum diagnostics over in_mask, the ROI estimates of roi = (labels[V], values), and the spatially
    regularised fit of spatial = (flat, shape, mu, n_sweeps) started from the point fit's fsol / status (host or CUDA):
    lambda_v from a second `t2_fit` with MET2_T2_FLAG_REG_IS_LAMBDA, the neighbour table of the fitted voxels, then the
    sweeps.  Returns ({"diagnostics", "roi"} as requested, the spatial fit's fsol / est_signal / maps / status as CUDA
    tensors); reg stays the point fit's."""
    extra, sp = {}, {}
    if in_mask is not None:
        extra["diagnostics"] = mean_spectrum_diagnostics(plan, sig, fa_index, in_mask, fsol_sum)
    if roi is not None:
        extra["roi"] = roi_estimates(plan, sig, fa_index, roi[0], roi[1])
    if spatial is not None:
        flat, shape, mu, n_sweeps = spatial
        lam = plan.t2_fit(sig, fa_index, flags=batched.REG_IS_LAMBDA)["reg"]
        status = torch.as_tensor(status).to(plan.dev)
        nbr, colours = spatial_neighbours(flat, shape, ((status & batched.ST_SKIPPED) == 0).cpu().numpy())
        sp = plan.spatial_fit(sig, fa_index, lam, fsol, nbr, colours, mu, n_sweeps, status=status)
        sp = {k: sp[k] for k in ("fsol", "est_signal", "maps", "status")}
    return extra, sp


class MultiGpuFit:
    """Steps 2-4 of ONE volume on several GPUs of one node, host memory in -> host memory out (the reference's only
    parallel knob, `num_cores` of motor_recon_met2 — joblib workers over image rows, motor...:165,357,365,435 — becomes
    the number of GPUs).  Voxels are independent, so there is no collective: the voxel list is dealt to the devices in
    a few large contiguous chunks (`chunk_deal`), each device copies its chunks from the (pinned) input array, runs the
    stages on its own stream and copies every output straight into its rows of ONE set of pinned host arrays —
    disjoint ranges, written by DMA, nothing to gather afterwards.  Per-voxel results are byte-identical to the
    single-GPU run (tests/test_gpu_multi.py, tests/test_gpu_pipeline.py)."""

    def __init__(self, plans, chunks_per_device=4):
        if not plans:
            raise ValueError("MultiGpuFit needs at least one plan")
        self.plans = list(plans)
        self.chunks_per_device = int(chunks_per_device)
        self.streams = [torch.cuda.Stream(device=p.dev) for p in self.plans]
        self._bufs = {}

    @classmethod
    def create(cls, n_gpus, *plan_args, chunks_per_device=4, **plan_kwargs):
        """One Met2Plan per device (built concurrently; each device computes its own dictionary and tables)."""
        avail = torch.cuda.device_count()
        if avail < 1:
            raise batched._lib.Met2Error("met2: no CUDA device available — this package has no CPU fallback")
        n = avail if n_gpus is None or n_gpus < 1 else min(int(n_gpus), avail)
        from concurrent.futures import ThreadPoolExecutor
        with ThreadPoolExecutor(max_workers=n) as ex:
            plans = list(ex.map(lambda d: batched.Met2Plan(*plan_args, device=torch.device("cuda", d), **plan_kwargs),
                                range(n)))
        return cls(plans, chunks_per_device)

    def fit(self, sig, sig_fa=None, out=None, n_bootstrap=0, bootstrap_seed=0, parametric=False, sigma=None):
        """sig[V, nTE] (+ sig_fa for the FA stage): host tensors / arrays, pinned for full-speed DMA.  `out`: dict of
        host tensors as from `host_buffers` (what it lacks is allocated).  Returns dict of numpy views of `out`.
        n_bootstrap > 0: also the per-voxel bootstrap of the maps (keys boot_*), each device over its own chunks with
        voxel_offset = the chunk's start, so the result does not depend on the device count.  parametric: also the
        three-pool parametric fit (keys param_*).  sigma[V] (host, raw signal units): also the Rician-likelihood fit
        (keys rician_*); each device copies its chunks of it beside sig.

        Everything is ENQUEUED from this one thread, phase by phase over the devices (copies in, then each stage of
        `_stages`, then copies out: ~0.1 ms of host time per device and phase, all asynchronous), then the streams are
        drained.  A thread per device was measured slower: two threads inside the CUDA runtime stalled each other for
        ~36 ms per call (profiles/r02_multi_gpu.json), a serial enqueue staggers the devices by well under a
        millisecond."""
        sig = torch.as_tensor(sig)
        if sig_fa is not None:
            sig_fa = torch.as_tensor(sig_fa)
        rician = sigma is not None
        if rician:
            sigma = torch.as_tensor(sigma, dtype=torch.float64)
        V = sig.shape[0]
        stages = _stages(False, n_bootstrap, bootstrap_seed, parametric, rician)
        names = [name for name, *_ in _outputs(stages)]
        if out is None or not all(k in out for k in names):
            out = {**host_buffers(self.plans[0], V, n_bootstrap=n_bootstrap, parametric=parametric, rician=rician),
                   **(out or {})}
        nd = len(self.plans)
        parts = chunk_deal(V, nd, self.chunks_per_device)
        trace = [dict() for _ in self.plans] if os.environ.get("MET2_MULTI_TRACE") else None
        t0 = time.perf_counter()

        def mark(d, what):
            if trace is not None:
                trace[d][what] = round(1e3 * (time.perf_counter() - t0), 2)
        live = [d for d in range(nd) if parts[d]]
        bufs = {}
        for d in live:                                   # ---- phase 1: host -> device
            plan = self.plans[d]
            Vd = sum(hi - lo for lo, hi in parts[d])
            key = (d, Vd, sig_fa is not None, rician)
            b = self._bufs.get(key)
            with torch.cuda.device(plan.dev), torch.cuda.stream(self.streams[d]):
                if b is None:
                    d_sig = torch.empty((Vd, plan.nTE), dtype=torch.float64, device=plan.dev)
                    b = dict(sig=d_sig, sig_fa=d_sig if sig_fa is None else torch.empty_like(d_sig), fa=None, t2=None,
                             sigma=torch.empty(Vd, dtype=torch.float64, device=plan.dev) if rician else None)
                    self._bufs = {k: v for k, v in self._bufs.items() if k[0] != d}
                    self._bufs[key] = b
                b["ranges"] = parts[d]
                o = 0
                for lo, hi in parts[d]:
                    b["sig"][o:o + hi - lo].copy_(sig[lo:hi], non_blocking=True)
                    if sig_fa is not None:
                        b["sig_fa"][o:o + hi - lo].copy_(sig_fa[lo:hi], non_blocking=True)
                    if rician:
                        b["sigma"][o:o + hi - lo].copy_(sigma[lo:hi], non_blocking=True)
                    o += hi - lo
            bufs[d] = b
            mark(d, "h2d_enqueued")
        res = {d: {} for d in live}
        for name, stage in stages:                       # ---- phases 2-3: each stage on every device
            for d in live:
                with torch.cuda.device(self.plans[d].dev), torch.cuda.stream(self.streams[d]):
                    res[d].update(stage(self.plans[d], bufs[d]))
                mark(d, name + "_enqueued")
        for d in live:                                   # ---- phase 4: device -> its rows of the host arrays
            with torch.cuda.device(self.plans[d].dev), torch.cuda.stream(self.streams[d]):
                o = 0
                for lo, hi in parts[d]:
                    for k in names:
                        out[k][lo:hi].copy_(res[d][k][o:o + hi - lo], non_blocking=True)
                    o += hi - lo
            mark(d, "d2h_enqueued")
        fs = torch.zeros(self.plans[0].npc, dtype=torch.float64)
        for d in live:                                   # ---- drain; fixed device order: deterministic fsol_sum
            self.streams[d].synchronize()
            mark(d, "stream_done")
            with torch.cuda.device(self.plans[d].dev), torch.cuda.stream(self.streams[d]):
                fs += bufs[d]["fa"]["fsol_sum"].cpu()
        out["fsol_sum"][:] = fs
        self.last_trace = trace
        return {k: (v.numpy() if k == "fsol_sum" else v[:V].numpy()) for k, v in out.items()}


def fit_voxels(plan, sig, sig_fa=None, pinned_out=None, in_mask=None, roi=None, fa_only=False, n_bootstrap=0,
               bootstrap_seed=0, voxel_offset=0, spatial=None, parametric=False, sigma=None):
    """Steps 2-4 on a list of voxels given as host array sig[V, nTE]; returns host arrays (dict).
    in_mask[V] (optional): also return the mean-spectrum diagnostics of motor...:375-403 over the voxels with
    in_mask == 1 (key "diagnostics").  roi = (labels[V], values) (optional): also the ROI-based estimates of
    motor_recon_met2_real_data_ROI.py:405-445 (key "roi").  n_bootstrap > 0: also the per-voxel bootstrap of the maps
    with that many replicates (keys boot_*); voxel_offset: the position of sig[0] in the whole voxel list (a torchrun
    rank's slab start).  spatial = (flat, shape, mu, n_sweeps) (optional): the voxels are the masked voxels flat[V] of
    a volume of `shape`, and fsol / est_signal / maps / status are those of the spatially regularised fit with coupling
    weight mu.  parametric: also the three-pool parametric fit started from the point fit (keys param_*).  sigma[V]
    (raw signal units): also the Rician-likelihood fit started from the point fit (keys rician_*).  fa_only: only the
    FA stage's outputs."""
    dev = plan.dev
    V = sig.shape[0]
    with torch.cuda.device(dev):
        d_sig = torch.as_tensor(sig).to(dev, non_blocking=True)
        if sig_fa is None:
            d_sig_fa = d_sig
        elif isinstance(sig_fa, torch.Tensor):
            d_sig_fa = sig_fa.to(dev)
        else:
            d_sig_fa = torch.as_tensor(sig_fa).to(dev, non_blocking=True)
        d_sigma = None if sigma is None else torch.as_tensor(sigma, dtype=torch.float64).to(dev, non_blocking=True)
        s = dict(sig=d_sig, sig_fa=d_sig_fa, sigma=d_sigma, ranges=[(voxel_offset, voxel_offset + V)], fa=None, t2=None)
        stages = _stages(fa_only, n_bootstrap, bootstrap_seed, parametric, sigma is not None)
        out = {}
        for _, stage in stages:
            out.update(stage(plan, s))
        out["fsol_sum"] = s["fa"]["fsol_sum"]
        extra = {}
        if V > 0:
            extra, sp = _whole_volume(plan, d_sig, out["fa_index"], out["fsol_sum"], in_mask, roi,
                                      None if fa_only else spatial, out.get("fsol"), out.get("status"))
            out.update(sp)
        host = {}
        for k in [name for name, *_ in _outputs(stages)] + ["fsol_sum"]:
            t = out[k]
            if pinned_out is not None and k in pinned_out:
                pinned_out[k][:t.shape[0]].copy_(t, non_blocking=True)
                host[k] = pinned_out[k][:t.shape[0]]
            else:
                host[k] = t.cpu()
        torch.cuda.synchronize(dev)
    res = {k: v.numpy() for k, v in host.items()}
    res.update(extra)
    return res


def recon_arrays(data, mask, TE_array, TR, reg_method, reg_matrix, FA_method, myelin_T2=40.0, data_fa=None, plan=None,
                 npc=None, n_alphas=None, device=None, rank=0, world_size=1, diagnostics=False, rois=None,
                 premasked=False, fa_only=False, n_gpus=1, n_bootstrap=0, bootstrap_seed=0, spatial_mu=0.0,
                 spatial_sweeps=10, parametric=False, rician_sigma=None):
    """Steps 2-4 of motor_recon_met2 on in-memory arrays.  Returns the ten output volumes (plus FA_index) as numpy.

    n_bootstrap > 0: also the per-voxel bootstrap uncertainty of the six maps with that many replicates per voxel
    (`batched.Met2Plan.bootstrap`): volumes "<MAP>_bootstrap" [nx, ny, nz, 4] (mean, sd, p2.5, p97.5) and
    "bootstrap_n_valid" [nx, ny, nz]; voxels outside the mask or skipped by the fit are zero.  Replicates are keyed on
    the voxel's position in the masked-voxel list and on bootstrap_seed, so the volumes are the same for any number of
    GPUs or ranks.

    spatial_mu > 0: the maps, fsol_4D, Est_Signal and status are those of the spatially regularised fit
    (`batched.Met2Plan.spatial_fit`, definition in csrc/met2_spatial.cu): spatial_sweeps red-black sweeps that couple
    each fitted voxel's spectrum to its fitted face neighbours with weight spatial_mu, started from the point fit; FA
    and reg_param stay the point fit's.  With several GPUs the point fit is spread over them and the sweeps run on the
    first.  It needs the whole volume in one process (world_size 1) and cannot be combined with n_bootstrap.

    parametric: also the three-pool parametric fit (`batched.Met2Plan.param_fit`, definition in csrc/met2_param.cu)
    started from each voxel's point fit: volumes MWF_3pool, IEWF_3pool, FWF_3pool, T2_M_3pool, T2_IE_3pool, T2_FW_3pool
    (each T2 is 0 where its pool's amplitude is 0), FA_3pool, TWC_3pool, SSE_3pool [nx, ny, nz] and Est_Signal_3pool
    [nx, ny, nz, nt]; zero outside the mask and where the point fit skipped the voxel.  The ten standard volumes are
    unchanged.  Per voxel, so it runs on every GPU and rank like the point fit; it cannot be combined with spatial_mu,
    since either spectrum could then start it.

    rician_sigma (a number or an [nx, ny, nz] array, the noise SD in the data's units): also the Rician-likelihood fit
    (`batched.Met2Plan.rician_fit`, definition in csrc/met2_rician.cu) started from each voxel's point fit, with the
    lambda that fit selected: volumes MWF_rician, IEWF_rician, FWF_rician, T2_M_rician, T2_IE_rician, TWC_rician,
    fsol_4D_rician, Est_Signal_rician and rician_iters (int32, MM solves run); zero outside the mask and where the
    point fit skipped the voxel or sigma is not finite and >= 0.  The ten standard volumes are unchanged.  Per voxel,
    so it runs on every GPU and rank like the point fit; it cannot be combined with spatial_mu.

    n_gpus != 1 (None / -1 = all visible GPUs): the voxel list of this ONE volume is spread over the GPUs of the node by
    `MultiGpuFit` (host in -> host out, no collective).  With world_size > 1 (one process per GPU under torchrun) only
    this rank's slab of the masked voxels is fitted and the other voxels are left zero; the caller combines the ranks
    (`gather_slabs`).  fa_only: stop after the flip-angle stage (the ROI-based estimator never fits voxel spectra,
    motor_recon_met2_real_data_ROI.py:349-445): the spectrum volumes are not produced.
    """
    spatial_mu = float(spatial_mu)
    if not (np.isfinite(spatial_mu) and spatial_mu >= 0.0):
        raise ValueError("spatial_mu must be finite and >= 0")
    if spatial_mu > 0 and world_size != 1:
        raise ValueError("the spatially regularised fit couples neighbouring voxels: run it unsharded")
    if spatial_mu > 0 and n_bootstrap > 0:
        raise ValueError("spatial_mu > 0 cannot be combined with n_bootstrap")
    if spatial_mu > 0 and parametric:
        raise ValueError("spatial_mu > 0 cannot be combined with parametric: it is ambiguous which spectrum starts the "
                         "parametric fit")
    if rician_sigma is not None and spatial_mu > 0:
        raise ValueError("spatial_mu > 0 cannot be combined with rician_sigma: it is ambiguous which spectrum starts the "
                         "Rician fit")
    data = np.asarray(data, dtype=np.float64)
    nx, ny, nz, nt = data.shape
    TE_array = np.asarray(TE_array, dtype=np.float64)
    multi = None
    if plan is None:
        plan_args = (TE_array.shape[0], TE_array[1] - TE_array[0], TR)
        plan_kw = dict(reg_method=reg_method, reg_matrix=reg_matrix, FA_method=FA_method, myelin_T2=myelin_T2, npc=npc,
                       n_alphas=n_alphas)
        want = torch.cuda.device_count() if (n_gpus is None or n_gpus < 1) else min(int(n_gpus), torch.cuda.device_count())
        if world_size == 1 and want > 1 and device is None and not fa_only:
            multi = MultiGpuFit.create(want, *plan_args, **plan_kw)
            plan = multi.plans[0]
        else:
            plan = batched.Met2Plan(*plan_args, device=device, **plan_kw)
    flat, sig = masked_voxel_list(data, mask, premasked)
    lo, hi = slab_bounds(len(flat), rank, world_size)
    sigma = None
    if rician_sigma is not None and not fa_only:
        sigma = np.broadcast_to(np.asarray(rician_sigma, dtype=np.float64), (nx, ny, nz)).reshape(-1)[flat[lo:hi]]
    sig_fa = None
    if data_fa is not None:
        if isinstance(data_fa, torch.Tensor):
            # smoothed volume already on the GPU (batched.gaussian_smooth): gather the slab's voxels there
            idx = torch.as_tensor(flat[lo:hi]).to(data_fa.device)
            sig_fa = data_fa.reshape(-1, nt).index_select(0, idx)
            if not premasked:
                m = torch.as_tensor(np.asarray(mask).reshape(-1)[flat[lo:hi]].astype(np.float64)).to(data_fa.device)
                sig_fa = (sig_fa * m[:, None]).clamp_min(0.0)
        else:
            _, sig_fa_all = masked_voxel_list(np.asarray(data_fa, dtype=np.float64), mask, premasked)
            sig_fa = sig_fa_all[lo:hi]
    if (diagnostics or rois is not None) and world_size != 1:
        raise ValueError("mean-spectrum diagnostics / ROI estimates are whole-volume reductions: run them unsharded")
    roi = None
    if rois is not None:
        # ROIs * mask, labels = np.unique without 0 (motor_recon_met2_real_data_ROI.py:166-183)
        rl = (np.asarray(rois).astype(np.int64) * np.asarray(mask).astype(np.int64)).reshape(-1)
        vals = np.unique(np.asarray(rois).astype(np.int64))
        roi = (rl[flat], vals[vals != 0])
    in_mask = np.asarray(mask).reshape(-1)[flat] if diagnostics else None
    spatial = (flat, (nx, ny, nz), spatial_mu, spatial_sweeps) if spatial_mu > 0 and not fa_only else None
    if multi is not None:
        V = hi - lo
        pin = torch.empty((V, nt), dtype=torch.float64).pin_memory()
        pin.numpy()[:] = sig[lo:hi]
        pin_fa = None
        if sig_fa is not None:
            pin_fa = torch.empty((V, nt), dtype=torch.float64).pin_memory()
            pin_fa.copy_(sig_fa if isinstance(sig_fa, torch.Tensor) else torch.as_tensor(sig_fa))
        pin_sigma = None
        if sigma is not None:
            pin_sigma = torch.empty(V, dtype=torch.float64).pin_memory()
            pin_sigma.numpy()[:] = sigma
        res = multi.fit(pin, pin_fa, n_bootstrap=n_bootstrap, bootstrap_seed=bootstrap_seed, parametric=parametric,
                        sigma=pin_sigma)
        if V > 0 and (in_mask is not None or roi is not None or spatial is not None):
            # these couple the voxels of every device's chunks: on the first device, from the gathered point fit
            with torch.cuda.device(plan.dev):
                d_sig = pin.to(plan.dev, non_blocking=True)
                d_idx = torch.as_tensor(res["fa_index"]).to(plan.dev)
                extra, sp = _whole_volume(plan, d_sig, d_idx, res["fsol_sum"], in_mask, roi, spatial, res["fsol"],
                                          res["status"])
                res.update(extra, **{k: v.cpu().numpy() for k, v in sp.items()})
    else:
        res = fit_voxels(plan, sig[lo:hi], sig_fa, in_mask=in_mask, roi=roi, fa_only=fa_only,
                         n_bootstrap=n_bootstrap, bootstrap_seed=bootstrap_seed, voxel_offset=lo, spatial=spatial,
                         parametric=parametric, sigma=sigma)
    sel = flat[lo:hi]
    vol = {}
    for name, key, col, dtype in VOLUMES:
        if key in res:
            src = res[key] if col is None else res[key][:, col]
            a = np.zeros((nx * ny * nz,) + src.shape[1:], dtype=dtype)
            a[sel] = src
            vol[name] = a.reshape((nx, ny, nz) + src.shape[1:])
    vol["mean_T2_dist"] = res["fsol_sum"]
    vol["T2s"] = plan.T2s
    vol.update({k: res[k] for k in ("diagnostics", "roi") if k in res})
    return vol


def gather_slabs(res, index, n_total, group=None):
    """Final gather of a one-process-per-GPU run (torchrun): `res` holds this rank's per-voxel outputs (arrays with
    leading dimension len(index)) for the voxels `index` (positions in the full voxel list of length n_total).  Every
    rank's rows are all-gathered — SLABS, padded to the longest one; never zero-padded full volumes — and placed at
    their positions.  NCCL for the CUDA build, gloo in the CPU test.  Returns full-length arrays on every rank."""
    import torch.distributed as dist
    index = np.asarray(index, dtype=np.int64)
    if not dist.is_initialized() or dist.get_world_size(group) == 1:
        out = {}
        for k, a in res.items():
            a = np.asarray(a)
            full = np.zeros((n_total,) + a.shape[1:], dtype=a.dtype)
            full[index] = a
            out[k] = full
        return out
    world = dist.get_world_size(group)
    use_cuda = dist.get_backend(group) == "nccl"
    dev = torch.device("cuda", torch.cuda.current_device()) if use_cuda else torch.device("cpu")
    counts = torch.zeros(world, dtype=torch.int64, device=dev)
    counts[dist.get_rank(group)] = len(index)
    dist.all_reduce(counts, group=group)
    counts = counts.cpu().numpy()
    nmax = int(counts.max())

    def gather(t):
        pad = torch.zeros((nmax,) + tuple(t.shape[1:]), dtype=t.dtype, device=dev)
        pad[:t.shape[0]] = t.to(dev)
        allt = torch.empty((world * nmax,) + tuple(t.shape[1:]), dtype=t.dtype, device=dev)
        dist.all_gather_into_tensor(allt, pad, group=group)
        return allt.reshape((world, nmax) + tuple(t.shape[1:]))
    idx_all = gather(torch.as_tensor(index)).cpu().numpy()
    out = {}
    for k, a in res.items():
        t = a if isinstance(a, torch.Tensor) else torch.as_tensor(np.ascontiguousarray(a))
        g = gather(t).cpu().numpy()
        full = np.zeros((n_total,) + g.shape[2:], dtype=g.dtype)
        for r in range(world):
            full[idx_all[r, :counts[r]]] = g[r, :counts[r]]
        out[k] = full
    return out


def _segment_x2(plan, mean_signal, mean_kernel, Laplac_plan, factor):
    """X2 fit (algorithms.py:211, no normalisation by M[0]) of every segment's mean signal against its mean kernel.
    ONE regularised fit (reg = the selected lambda) and one plain NNLS fit; k_est = SSE(lambda) / SSE(plain)
    (algorithms.py:231-233) follows from the two fitted signals.  Returns (dictionary, idx, x2 fit, nnls fit, k_est)."""
    d = batched.Dictionary.from_device(mean_kernel)
    idx = torch.arange(mean_signal.shape[0], dtype=torch.int32, device=mean_signal.device)
    x2 = Laplac_plan.t2_fit(mean_signal, idx, reg_method="X2", flags=3, dictionary=d, factor=float(factor))
    nn = Laplac_plan.t2_fit(mean_signal, idx, reg_method="NNLS", flags=2, dictionary=d)
    sse = ((x2["est_signal"] - mean_signal) ** 2).sum(dim=1)
    sse0 = ((nn["est_signal"] - mean_signal) ** 2).sum(dim=1)
    return d, idx, x2, nn, sse / sse0


def mean_spectrum_diagnostics(plan, sig, fa_index, in_mask, fsol_sum, factor=1.01):
    """The three curves of the reference's 'Mean_spectrum_from_all_voxels' figure (motor...:375-403):
    mean_T2_dist (normalised sum of the FA-stage NNLS spectra), dist_T2_mean1 (NNLS of the mask-mean signal against the
    mask-mean kernel) and dist_T2_mean2 (X2 with factor 1.01 and the identity matrix on the same pair).
    sig[V, nTE] / fa_index[V] on the GPU; in_mask[V]: 1 where the reference's `mask == 1` test holds."""
    dev = plan.dev
    labels = torch.as_tensor(np.asarray(in_mask)).to(dev) if not isinstance(in_mask, torch.Tensor) else in_mask.to(dev)
    labels = torch.where(labels == 1, 0, -1).to(torch.int32)
    msig, mker, counts = batched.segment_means(sig, fa_index, labels, 1, plan.dict_hr)
    plan_I = plan if np.array_equal(plan.Laplac, np.eye(plan.npc)) else batched.Met2Plan(
        plan.nTE, plan.tau, plan.TR, reg_method="X2", reg_matrix="I", FA_method="brute-force", npc=plan.npc,
        Dic_3D=np.zeros((plan.nTE, plan.npc, 1)), T2s=plan.T2s, device=dev)
    d, idx, x2, nn, k_est = _segment_x2(plan, msig, mker, plan_I, factor)
    f1 = nn["fsol"][0].cpu().numpy()
    f2 = x2["fsol"][0].cpu().numpy()
    fs = np.asarray(fsol_sum.cpu().numpy() if isinstance(fsol_sum, torch.Tensor) else fsol_sum, dtype=np.float64)
    with np.errstate(all="ignore"):
        return dict(T2s=plan.T2s, mean_T2_dist=fs / np.sum(fs), dist_T2_mean1=f1 / np.sum(f1),
                    dist_T2_mean2=f2 / np.sum(f2), total_signal=msig[0].cpu().numpy(),
                    total_Kernel=mker[0].cpu().numpy(), nv=int(counts[0]), reg_opt2=float(x2["reg"][0]),
                    k_est=float(k_est[0]))


def roi_estimates(plan, sig, fa_index, roi_labels, roi_values, factor=1.01):
    """ROI-based estimator of motor/motor_recon_met2_real_data_ROI.py:405-445: for every ROI value, X2 (factor 1.01,
    the plan's regularisation matrix) of the ROI-mean signal against the ROI-mean kernel, then the Step-4 metrics of the
    normalised spectrum.  sig[V, nTE], fa_index[V], roi_labels[V] (integer label per voxel), roi_values: the labels to
    report (np.unique(ROIs) without 0 in the reference).  Returns host arrays: fsol_ROIs[nROI, nT2] (normalised),
    MWF/IEWF/FWF/T2M/T2IE/TWC[nROI], reg_opt[nROI], k_est[nROI], counts[nROI]."""
    dev = plan.dev
    roi_values = np.asarray(roi_values).astype(np.int64)
    lab = roi_labels if isinstance(roi_labels, torch.Tensor) else torch.as_tensor(np.asarray(roi_labels).astype(np.int64))
    lab = lab.to(dev).to(torch.int64)
    # label value -> segment id (position in roi_values); everything else -> -1
    seg = torch.full_like(lab, -1)
    for i, val in enumerate(roi_values.tolist()):
        seg = torch.where(lab == val, i, seg)
    n = len(roi_values)
    msig, mker, counts = batched.segment_means(sig, fa_index, seg.to(torch.int32), n, plan.dict_hr)
    d, idx, x2, nn, k_est = _segment_x2(plan, msig, mker, plan, factor)
    maps = x2["maps"].cpu().numpy()
    f = x2["fsol"].cpu().numpy()
    vt = maps[:, 5]
    return dict(roi_values=roi_values, fsol_ROIs=f / vt[:, None], MWF_ROIs=maps[:, 0], IEWF_ROIs=maps[:, 1],
                FWF_ROIs=maps[:, 2], T2M_ROIs=maps[:, 3], T2IE_ROIs=maps[:, 4], TWC_ROIs=vt,
                reg_opt=x2["reg"].cpu().numpy(), k_est=k_est.cpu().numpy(), counts=counts.cpu().numpy(),
                mean_signal=msig.cpu().numpy(), mean_kernel=mker.cpu().numpy())
