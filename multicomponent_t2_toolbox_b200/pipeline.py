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


OUT_KEYS = ("fa_index", "fa_deg", "km", "fa_status", "fsol", "est_signal", "reg", "maps", "status")
BOOT_KEYS = ("boot_stats", "boot_n_valid")


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


SPATIAL_KEYS = ("fsol", "est_signal", "maps", "status")


def spatial_fitted(plan, sig, fa_index, t2, flat, shape, mu, n_sweeps):
    """`Met2Plan.spatial_fit` after the point fit `t2` (the `t2_fit` result on sig[V, nTE] at fa_index[V], CUDA) of the
    masked voxels flat[V] of a volume of `shape`: lambda_v from a second `t2_fit` with MET2_T2_FLAG_REG_IS_LAMBDA, the
    neighbour table of the fitted voxels (`spatial_neighbours`; reads the point fit's status back to the host), then the
    sweeps.  Returns dict(fsol, est_signal, maps, status) of CUDA tensors; reg stays the point fit's."""
    lam = plan.t2_fit(sig, fa_index, flags=batched.REG_IS_LAMBDA)["reg"]
    fitted = ((t2["status"] & batched.ST_SKIPPED) == 0).cpu().numpy()
    nbr, colours = spatial_neighbours(flat, shape, fitted)
    sp = plan.spatial_fit(sig, fa_index, lam, t2["fsol"], nbr, colours, mu, n_sweeps, status=t2["status"])
    return {k: sp[k] for k in SPATIAL_KEYS}


def bootstrap_fitted(plan, sig, fa_index, t2, n_bootstrap, seed, voxel_offset):
    """`Met2Plan.bootstrap` of the voxels of one point fit (`t2`: the `t2_fit` result on sig[V, nTE] at fa_index[V]),
    with voxel_offset = the position of sig[0] in the whole voxel list.  Voxels the point fit skipped get zeros, like
    their maps.  Returns dict(boot_stats[V, 6, 4], boot_n_valid[V]) of CUDA tensors, enqueued on the current stream."""
    stats, n_valid = plan.bootstrap(sig, fa_index, t2["est_signal"], B=n_bootstrap, seed=seed,
                                    voxel_offset=voxel_offset)
    skipped = (t2["status"] & batched.ST_SKIPPED) != 0
    stats.masked_fill_(skipped[:, None, None], 0.0)
    n_valid.masked_fill_(skipped, 0)
    return dict(boot_stats=stats, boot_n_valid=n_valid)


PARAM_KEYS = ("param_params", "param_maps", "param_est_signal", "param_sse", "param_iters", "param_status")
# the volumes of the three-pool parametric fit: name -> (output, column)
PARAM_VOLUMES = {"MWF_3pool": ("param_maps", 0), "IEWF_3pool": ("param_maps", 1), "FWF_3pool": ("param_maps", 2),
                 "T2_M_3pool": ("param_maps", 3), "T2_IE_3pool": ("param_maps", 4), "T2_FW_3pool": ("param_params", 5),
                 "FA_3pool": ("param_params", 6), "TWC_3pool": ("param_maps", 5), "SSE_3pool": ("param_sse", None),
                 "Est_Signal_3pool": ("param_est_signal", None)}


def param_fitted(plan, sig, fa_deg, t2):
    """`Met2Plan.param_fit` started from one point fit (`t2`: the `t2_fit` result on sig[V, nTE]; fa_deg[V] the FA
    stage's angles).  Returns the PARAM_KEYS of CUDA tensors, enqueued on the current stream; T2_FW (params column 5)
    is zeroed where the free-water amplitude is 0, like T2_M and T2_IE in the maps."""
    pf = plan.param_fit(sig, fa_deg, t2["fsol"], t2["status"])
    pf["params"][:, 5].masked_fill_(pf["params"][:, 2] <= 0.0, 0.0)
    return {"param_" + k: pf[k] for k in ("params", "maps", "est_signal", "sse", "iters", "status")}


def host_buffers(plan, V, pinned=True):
    """Host (pinned) arrays for the per-voxel outputs of `fit_voxels` / `MultiGpuFit.fit` of V voxels."""
    def mk(shape, dtype):
        t = torch.empty(shape, dtype=dtype)
        return t.pin_memory() if pinned and torch.cuda.is_available() else t
    return {"fsol": mk((V, plan.npc), torch.float64), "est_signal": mk((V, plan.nTE), torch.float64),
            "maps": mk((V, 6), torch.float64), "reg": mk((V,), torch.float64), "fa_deg": mk((V,), torch.float64),
            "fa_index": mk((V,), torch.int32), "km": mk((V,), torch.float64), "status": mk((V,), torch.int32),
            "fa_status": mk((V,), torch.int32), "fsol_sum": mk((plan.npc,), torch.float64)}


class MultiGpuFit:
    """Steps 2-4 of ONE volume on several GPUs of one node, host memory in -> host memory out (the reference's only
    parallel knob, `num_cores` of motor_recon_met2 — joblib workers over image rows, motor...:165,357,365,435 — becomes
    the number of GPUs).  Voxels are independent, so there is no collective: the voxel list is dealt to the devices in
    a few large contiguous chunks (`chunk_deal`), one host thread per device copies its chunks from the (pinned) input
    array, runs the two batched kernels on its own stream and copies every output straight into its rows of ONE set of
    pinned host arrays — disjoint ranges, written by DMA, nothing to gather afterwards.  Per-voxel results are
    byte-identical to the single-GPU run (tests/test_gpu_multi.py)."""

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

    def fit(self, sig, sig_fa=None, out=None, n_bootstrap=0, bootstrap_seed=0, parametric=False):
        """sig[V, nTE] (+ sig_fa for the FA stage): host tensors / arrays, pinned for full-speed DMA.  `out`: dict of
        host tensors as from `host_buffers` (allocated if None).  Returns dict of numpy views of `out`.
        n_bootstrap > 0: also the per-voxel bootstrap of the maps (`bootstrap_fitted`, keys BOOT_KEYS), each device
        over its own chunks with voxel_offset = the chunk's start, so the result does not depend on the device count.
        parametric: also the three-pool parametric fit (`param_fitted`, keys PARAM_KEYS), chunk by chunk on each device.

        Everything is ENQUEUED from this one thread, phase by phase over the devices (copies in, FA stage, T2 stage,
        copies out: ~0.1 ms of host time per device and phase, all asynchronous), then the streams are drained.  A
        thread per device was measured slower: two threads inside the CUDA runtime stalled each other for ~36 ms per
        call (profiles/r02_multi_gpu.json), a serial enqueue staggers the devices by well under a millisecond."""
        sig = torch.as_tensor(sig)
        if sig_fa is not None:
            sig_fa = torch.as_tensor(sig_fa)
        V = sig.shape[0]
        if out is None:
            out = host_buffers(self.plans[0], V)
        if n_bootstrap > 0 and "boot_stats" not in out:
            pin = torch.cuda.is_available()
            out["boot_stats"] = torch.empty((V, 6, 4), dtype=torch.float64, pin_memory=pin)
            out["boot_n_valid"] = torch.empty(V, dtype=torch.int32, pin_memory=pin)
        if parametric and "param_params" not in out:
            pin = torch.cuda.is_available()
            nTE = self.plans[0].nTE
            for k, shape, dt in (("param_params", (V, 7), torch.float64), ("param_maps", (V, 6), torch.float64),
                                 ("param_est_signal", (V, nTE), torch.float64), ("param_sse", (V,), torch.float64),
                                 ("param_iters", (V,), torch.int32), ("param_status", (V,), torch.int32)):
                out[k] = torch.empty(shape, dtype=dt, pin_memory=pin)
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
            key = (d, Vd, sig_fa is not None)
            b = self._bufs.get(key)
            with torch.cuda.device(plan.dev), torch.cuda.stream(self.streams[d]):
                if b is None:
                    b = dict(sig=torch.empty((Vd, plan.nTE), dtype=torch.float64, device=plan.dev),
                             sig_fa=(torch.empty((Vd, plan.nTE), dtype=torch.float64, device=plan.dev)
                                     if sig_fa is not None else None), fa=None, t2=None)
                    self._bufs = {k: v for k, v in self._bufs.items() if k[0] != d}
                    self._bufs[key] = b
                o = 0
                for lo, hi in parts[d]:
                    b["sig"][o:o + hi - lo].copy_(sig[lo:hi], non_blocking=True)
                    if sig_fa is not None:
                        b["sig_fa"][o:o + hi - lo].copy_(sig_fa[lo:hi], non_blocking=True)
                    o += hi - lo
            bufs[d] = b
            mark(d, "h2d_enqueued")
        for d in live:                                   # ---- phase 2: flip-angle stage
            plan, b = self.plans[d], bufs[d]
            with torch.cuda.device(plan.dev), torch.cuda.stream(self.streams[d]):
                b["fa"] = plan.fa_fit(b["sig"] if sig_fa is None else b["sig_fa"], out=b["fa"])
            mark(d, "fa_enqueued")
        for d in live:                                   # ---- phase 3: spectrum fit + maps
            plan, b = self.plans[d], bufs[d]
            with torch.cuda.device(plan.dev), torch.cuda.stream(self.streams[d]):
                b["t2"] = plan.t2_fit(b["sig"], b["fa"]["fa_index"], out=b["t2"])
            mark(d, "t2_enqueued")
        boot = {}
        if n_bootstrap > 0:
            for d in live:                               # ---- phase 3b: bootstrap, chunk by chunk
                plan, b = self.plans[d], bufs[d]
                with torch.cuda.device(plan.dev), torch.cuda.stream(self.streams[d]):
                    o, boot[d] = 0, []
                    for lo, hi in parts[d]:
                        rows = slice(o, o + hi - lo)
                        t2 = {k: b["t2"][k][rows] for k in ("est_signal", "status")}
                        boot[d].append(bootstrap_fitted(plan, b["sig"][rows], b["fa"]["fa_index"][rows], t2,
                                                        n_bootstrap, bootstrap_seed, lo))
                        o += hi - lo
                mark(d, "bootstrap_enqueued")
        par = {}
        if parametric:
            for d in live:                               # ---- phase 3c: parametric fit, chunk by chunk
                plan, b = self.plans[d], bufs[d]
                with torch.cuda.device(plan.dev), torch.cuda.stream(self.streams[d]):
                    o, par[d] = 0, []
                    for lo, hi in parts[d]:
                        rows = slice(o, o + hi - lo)
                        t2 = {k: b["t2"][k][rows] for k in ("fsol", "status")}
                        par[d].append(param_fitted(plan, b["sig"][rows], b["fa"]["fa_deg"][rows], t2))
                        o += hi - lo
                mark(d, "parametric_enqueued")
        for d in live:                                   # ---- phase 4: device -> its rows of the host arrays
            plan, b = self.plans[d], bufs[d]
            fa, t2 = b["fa"], b["t2"]
            dev_out = dict(fa_index=fa["fa_index"], fa_deg=fa["fa_deg"], km=fa["km"], fa_status=fa["status"],
                           fsol=t2["fsol"], est_signal=t2["est_signal"], reg=t2["reg"], maps=t2["maps"],
                           status=t2["status"])
            with torch.cuda.device(plan.dev), torch.cuda.stream(self.streams[d]):
                o = 0
                for i, (lo, hi) in enumerate(parts[d]):
                    for k in OUT_KEYS:
                        out[k][lo:hi].copy_(dev_out[k][o:o + hi - lo], non_blocking=True)
                    for k in (BOOT_KEYS if n_bootstrap > 0 else ()):
                        out[k][lo:hi].copy_(boot[d][i][k], non_blocking=True)
                    for k in (PARAM_KEYS if parametric else ()):
                        out[k][lo:hi].copy_(par[d][i][k], non_blocking=True)
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
               bootstrap_seed=0, voxel_offset=0, spatial=None, parametric=False):
    """Steps 2-4 on a list of voxels given as host array sig[V, nTE]; returns host arrays (dict).
    in_mask[V] (optional): also return the mean-spectrum diagnostics of motor...:375-403 over the voxels with
    in_mask == 1 (key "diagnostics").  roi = (labels[V], values) (optional): also the ROI-based estimates of
    motor_recon_met2_real_data_ROI.py:405-445 (key "roi").  n_bootstrap > 0: also the per-voxel bootstrap of the maps
    with that many replicates (`bootstrap_fitted`, keys BOOT_KEYS); voxel_offset: the position of sig[0] in the whole
    voxel list (a torchrun rank's slab start).  spatial = (flat, shape, mu, n_sweeps) (optional): the voxels are the
    masked voxels flat[V] of a volume of `shape`, and fsol / est_signal / maps / status are those of the spatially
    regularised fit with coupling weight mu (`spatial_fitted`).  parametric: also the three-pool parametric fit started
    from the point fit (`param_fitted`, keys PARAM_KEYS)."""
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
        fa = plan.fa_fit(d_sig_fa)
        out = dict(fa_index=fa["fa_index"], fa_deg=fa["fa_deg"], km=fa["km"], fsol_sum=fa["fsol_sum"],
                   fa_status=fa["status"])
        if not fa_only:
            t2 = plan.t2_fit(d_sig, fa["fa_index"])
            out.update(fsol=t2["fsol"], est_signal=t2["est_signal"], reg=t2["reg"], maps=t2["maps"], status=t2["status"])
            if spatial is not None:
                out.update(spatial_fitted(plan, d_sig, fa["fa_index"], t2, *spatial))
            if n_bootstrap > 0:
                out.update(bootstrap_fitted(plan, d_sig, fa["fa_index"], t2, n_bootstrap, bootstrap_seed, voxel_offset))
            if parametric:
                out.update(param_fitted(plan, d_sig, fa["fa_deg"], t2))
        extra = {}
        if in_mask is not None and V > 0:
            extra["diagnostics"] = mean_spectrum_diagnostics(plan, d_sig, fa["fa_index"], in_mask, fa["fsol_sum"])
        if roi is not None and V > 0:
            extra["roi"] = roi_estimates(plan, d_sig, fa["fa_index"], roi[0], roi[1])
        host = {}
        for k, t in out.items():
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
                 spatial_sweeps=10, parametric=False):
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
    if multi is not None:
        V = hi - lo
        pin = torch.empty((V, nt), dtype=torch.float64).pin_memory()
        pin.numpy()[:] = sig[lo:hi]
        pin_fa = None
        if sig_fa is not None:
            pin_fa = torch.empty((V, nt), dtype=torch.float64).pin_memory()
            pin_fa.copy_(sig_fa if isinstance(sig_fa, torch.Tensor) else torch.as_tensor(sig_fa))
        res = multi.fit(pin, pin_fa, n_bootstrap=n_bootstrap, bootstrap_seed=bootstrap_seed, parametric=parametric)
        if (in_mask is not None or roi is not None) and V > 0:
            # whole-volume reductions (a few ms): on the first device, from the gathered FA indices
            with torch.cuda.device(plan.dev):
                d_sig = pin.to(plan.dev, non_blocking=True)
                d_idx = torch.as_tensor(res["fa_index"]).to(plan.dev)
                if in_mask is not None:
                    res["diagnostics"] = mean_spectrum_diagnostics(plan, d_sig, d_idx, in_mask, res["fsol_sum"])
                if roi is not None:
                    res["roi"] = roi_estimates(plan, d_sig, d_idx, roi[0], roi[1])
        if spatial_mu > 0 and V > 0:
            # the sweeps couple voxels of every device's chunks: on the first device, from the gathered point fit
            with torch.cuda.device(plan.dev):
                d_sig = pin.to(plan.dev, non_blocking=True)
                d_idx = torch.as_tensor(res["fa_index"]).to(plan.dev)
                t2 = dict(fsol=torch.as_tensor(res["fsol"]).to(plan.dev),
                          status=torch.as_tensor(res["status"]).to(plan.dev))
                sp = spatial_fitted(plan, d_sig, d_idx, t2, flat, (nx, ny, nz), spatial_mu, spatial_sweeps)
                res.update({k: v.cpu().numpy() for k, v in sp.items()})
    else:
        spatial = (flat, (nx, ny, nz), spatial_mu, spatial_sweeps) if spatial_mu > 0 and not fa_only else None
        res = fit_voxels(plan, sig[lo:hi], sig_fa, in_mask=in_mask, roi=roi, fa_only=fa_only,
                         n_bootstrap=n_bootstrap, bootstrap_seed=bootstrap_seed, voxel_offset=lo, spatial=spatial,
                         parametric=parametric)
    sel = flat[lo:hi]
    nvox = nx * ny * nz
    vol = {}
    for name, key in (("FA", "fa_deg"), ("FA_index", "fa_index")):
        a = np.zeros(nvox)
        a[sel] = res[key]
        vol[name] = a.reshape(nx, ny, nz)
    vol["mean_T2_dist"] = res["fsol_sum"]
    vol["T2s"] = plan.T2s
    for k in ("diagnostics", "roi"):
        if k in res:
            vol[k] = res[k]
    if fa_only:
        return vol
    for i, name in enumerate(MAP_NAMES):
        a = np.zeros(nvox)
        a[sel] = res["maps"][:, i]
        vol[name] = a.reshape(nx, ny, nz)
    a = np.zeros(nvox)
    a[sel] = res["reg"]
    vol["reg_param"] = a.reshape(nx, ny, nz)
    f4 = np.zeros((nvox, plan.npc))
    f4[sel] = res["fsol"]
    vol["fsol_4D"] = f4.reshape(nx, ny, nz, plan.npc)
    s4 = np.zeros((nvox, nt))
    s4[sel] = res["est_signal"]
    vol["Est_Signal"] = s4.reshape(nx, ny, nz, nt)
    vol["status"] = np.zeros(nvox, dtype=np.int32)
    vol["status"][sel] = res["status"]
    vol["status"] = vol["status"].reshape(nx, ny, nz)
    if n_bootstrap > 0:
        for i, name in enumerate(MAP_NAMES):
            a = np.zeros((nvox, 4))
            a[sel] = res["boot_stats"][:, i, :]
            vol[name + "_bootstrap"] = a.reshape(nx, ny, nz, 4)
        a = np.zeros(nvox, dtype=np.int32)
        a[sel] = res["boot_n_valid"]
        vol["bootstrap_n_valid"] = a.reshape(nx, ny, nz)
    if parametric:
        for name, (key, col) in PARAM_VOLUMES.items():
            src = res[key] if col is None else res[key][:, col]
            a = np.zeros((nvox,) + src.shape[1:])
            a[sel] = src
            vol[name] = a.reshape((nx, ny, nz) + src.shape[1:])
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
