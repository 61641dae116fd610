#!/usr/bin/env python
"""bench.py — headline benchmark of the per-voxel MET2 inverse-problem path (BASELINE.json metric).

One "step" = one pass of the hot path (flip-angle estimation + regularised NNLS fit + maps; Steps 2+3+4 of
motor/motor_recon_met2_real_data.py) over one synthetic whole-brain volume: BASELINE.json configs[1] =
96x96x60 (552 960 voxels), nTE=32, 60 T2 bins, reg_method=X2 (factor 1.02), reg_matrix=I, FA_method=spline.
With N GPUs every rank fits its own volume of that size (weak scaling, no data-path collective; SURVEY.md §8e); the
north-star case — ONE volume over N GPUs, host memory in -> host memory out — is measured beside it (`one_volume`).

  python bench.py [--gpus N] [--steps K] [--warmup W]                 our CUDA path
  python bench.py ... --dump-outputs DIR                              + the outputs of the last timed step, DIR/*.npy
  python bench.py --impl reference [--gpus N] --steps K --warmup W    the reference's CPU algorithm (oracle port, all
                                                                      host cores, bounded sample per step)
Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import platform
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the checkout may be read-only: no __pycache__ next to the sources

METRIC = "fitted voxels/s (FA+reg NNLS)"
UNIT = "voxels/s"
SHAPE = (96, 96, 60)
N_ECHOES, TAU, TR = 32, 10.0, 1000.0
REG_METHOD, REG_MATRIX, FA_METHOD = "X2", "I", "spline"
WORKLOAD = "config2: synthetic brain 96x96x60 (552960 voxels), nTE=32, 60 T2, FA spline (15 knots -> 273 grid) + X2-I"
CONFIG = {"workload": WORKLOAD, "reg_method": REG_METHOD, "reg_matrix": REG_MATRIX, "FA_method": FA_METHOD,
          "nTE": N_ECHOES, "nT2": 60, "voxels_per_volume": SHAPE[0] * SHAPE[1] * SHAPE[2]}   # identical in both arms

FP64_PEAK_TFLOPS = 34.16    # own DFMA micro-benchmark on this pool's B200 (profiles/r01_fp64_peak_microbench.json);
                            # MEASURED_PEAKS.json has no FP64 entry
HBM_BYTES_PER_VOXEL_T2 = 32 * 8 + 4 + 60 * 8 + 32 * 8 + 8 + 6 * 8 + 4   # T2 kernel: read signal+index, write outputs
HBM_BYTES_PER_VOXEL_FA = 16 * 32 * 8 + 15 * 8 + 3 * 8 + 8                # FA kernels: signal per search angle + outputs
NCU_RECORD = "profiles/r02_kernel_counters.json"   # executed flops / DRAM traffic per voxel of the current kernels (ncu)
# --dump-outputs: per-voxel outputs at a fixed sample of this many voxels (104 float64 outputs + the voxel's index at
# the config-2 widths = 55 MB), so that the dump stays under 64 MB
DUMP_VOXELS = 65536


def f_alg():
    """Algorithmic (reference-formulation) flops per voxel, SURVEY.md §8(d): Lawson-Hanson QR on [D; sqrt(lambda) L]
    counted by oracle/flop_model.py (instrumented lh_nnls) on voxels of this workload; oracle/F_ALG.json."""
    with open(os.path.join(ROOT, "oracle", "F_ALG.json")) as fh:
        return json.load(fh)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--shape", default=None, help="override volume, e.g. 16,16,4 (debug only)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--t2-flags", type=int, default=0, help="extra MET2_T2_FLAG_* bits for every T2 fit (A/B runs only)")
    ap.add_argument("--gram", action="store_true",
                    help="A/B runs only: Gram-domain T2 kernel instead of the default reduced-echo-space kernel")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed (rank 0) as DIR/<name>.npy, float64: "
                         "FA and T2 outputs at a fixed, seeded sample of %d voxels (voxel_index.npy), fsol_sum whole"
                         % DUMP_VOXELS)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


# ---------------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows = []
        self.proc = None
        self.gpu = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return None
        time.sleep(0.15)
        self.proc.terminate()
        sm, reasons, smax = [], set(), None
        for ts, line in self.rows:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                smax = float(parts[2])
                if t0 - 0.05 <= ts <= t1 + 0.15:
                    sm.append(float(parts[1]))
                    for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"),
                                         parts[5:9]):
                        if val.lower().startswith("active"):
                            reasons.add(name)
            except ValueError:
                continue
        if not sm:
            all_sm = []
            for ts, line in self.rows:
                parts = [p.strip() for p in line.split(",")]
                try:
                    all_sm.append(float(parts[1]))
                except (ValueError, IndexError):
                    pass
            sm = all_sm[-3:]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------- CPU arms
_CPU_STATE = {}
CPU_SAMPLE_ROWS = 192          # 96 x 192 x 1 = 18 432 voxels per CPU step: 12 image rows per process on 16 cores


def cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return platform.processor() or "unknown"


def cpu_setup():
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import multiprocessing

    import met2_oracle as O
    if "dic" not in _CPU_STATE:
        g = O._grids(REG_METHOD, REG_MATRIX, FA_METHOD, 40.0, N_ECHOES, TAU, TR)
        # the dictionary is set-up, not the per-voxel path: build it once outside the timed region
        _CPU_STATE["dic"] = O.create_Dic_3D(g["npc"], g["T2s"], g["T1s"], N_ECHOES, TAU, g["alpha_values"], TR)
        _CPU_STATE["dic_lr"] = O.create_Dic_3D(g["npc"], g["T2s"], g["T1s"], N_ECHOES, TAU, g["alpha_spline"], TR)
        _CPU_STATE["cores"] = os.cpu_count() or 1
        _CPU_STATE["pool"] = multiprocessing.Pool(_CPU_STATE["cores"])
    return O


def cpu_run(rows, seed):
    """One bounded-sample pass of the reference algorithm on all host cores over a 96 x rows x 1 slab of the config-2
    phantom (image rows dealt to a process pool, like the reference's joblib loops); returns (voxels, seconds)."""
    O = cpu_setup()
    from multicomponent_t2_toolbox_b200.phantom import make_phantom
    nx = 96
    ph = make_phantom((nx, int(rows), 1), n_echoes=N_ECHOES, tau=TAU, TR=TR, seed=seed, fa_mode="b1")
    t0 = time.perf_counter()
    O.recon_volume(ph["data"], ph["mask"], ph["TE_array"], TR, REG_METHOD, REG_MATRIX, FA_METHOD, 40.0,
                   num_cores=_CPU_STATE["cores"], Dic_3D=_CPU_STATE["dic"], Dic_3D_LR=_CPU_STATE["dic_lr"],
                   pool=_CPU_STATE["pool"])
    dt = time.perf_counter() - t0
    return nx * int(rows), dt


def cpu_env():
    return {"cores": _CPU_STATE["cores"], "cpu_model": cpu_model(), "OMP_NUM_THREADS": os.environ.get("OMP_NUM_THREADS"),
            "kind": "port"}


def run_reference(args):
    """The reference's own CPU algorithm for the path (oracle port: bitwise equal to the unmodified reference,
    tests/test_oracle_vs_reference.py; /root/reference itself is not on the GPU box) on all host cores.  Every step is
    a 18 432-voxel slab (>= 73 728 voxels over the run, BASELINE.md §2) unless the whole run would exceed ~4.5 min."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    os.environ.setdefault("OMP_NUM_THREADS", "1")      # one BLAS thread per worker process (BASELINE.md §2)
    cpu_setup()
    nvox, dt = cpu_run(32, seed=100)                     # pilot to size the steps
    rate = nvox / dt
    total = max(1, args.steps + args.warmup)
    rows = CPU_SAMPLE_ROWS
    if total * 96 * rows / rate > 270.0:
        rows = int(max(48, min(CPU_SAMPLE_ROWS, (270.0 * rate / total) // (96 * 16) * 16)))
    for w in range(args.warmup):
        cpu_run(rows, seed=200 + w)
    t_total, v_total = 0.0, 0
    for k in range(args.steps):
        v, dt = cpu_run(rows, seed=300 + k)
        v_total += v
        t_total += dt
    value = v_total / t_total
    sample = "%d voxels/step (96x%dx1 slab of the config-2 phantom), %d steps = %d voxels" % (
        96 * rows, rows, args.steps, v_total)
    cb = dict(cpu_env(), value=value, unit=UNIT, sample=sample)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_total / max(1, args.steps),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": CONFIG,
            "note": "reference algorithm (oracle port of the reference's Python + SciPy Lawson-Hanson path, "
                    "multiprocessing over image rows with a persistent pool and a prebuilt dictionary)",
            "cpu_baseline": cb,
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)
    _CPU_STATE["pool"].close()
    return 0


# ---------------------------------------------------------------------------------------------------- our arm
def _ncu_record():
    try:
        with open(os.path.join(ROOT, NCU_RECORD)) as fh:
            return json.load(fh)
    except Exception:
        return {}


def _hbm_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            return json.load(fh)["hbm_gbs"], "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def run_ours(args):
    import torch
    import torch.distributed as dist

    from multicomponent_t2_toolbox_b200 import _lib, batched, pipeline
    from multicomponent_t2_toolbox_b200.phantom import make_phantom

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    json_fd = None
    host_group = None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL prints its version banner on stdout at communicator creation: point fd 1 at stderr for the duration of
        # the run and keep the original stdout for the one JSON line
        sys.stdout.flush()
        json_fd = os.dup(1)
        os.dup2(2, 1)
        dist.init_process_group("nccl", device_id=dev)
        host_group = dist.new_group(backend="gloo")     # host-side waits that leave the GPUs idle
    shape = SHAPE if args.shape is None else tuple(int(x) for x in args.shape.split(","))
    lib = _lib.load(build_if_missing=False)      # the library build() left in the tree; never rebuilt here

    ph = make_phantom(shape, n_echoes=N_ECHOES, tau=TAU, TR=TR, seed=2 + rank, fa_mode="b1", backend="gpu")
    sig_host = torch.as_tensor(ph["data"].reshape(-1, N_ECHOES)).pin_memory()
    V = sig_host.shape[0]
    plan = batched.Met2Plan(N_ECHOES, TAU, TR, reg_method=REG_METHOD, reg_matrix=REG_MATRIX, FA_method=FA_METHOD,
                            device=dev, t2_flags=args.t2_flags, echo_space=not args.gram)
    sig = sig_host.to(dev)
    fa_out = t2_out = None

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    n_warm = max(3, args.warmup)
    for _ in range(n_warm):
        fa_out = plan.fa_fit(sig, out=fa_out)
        t2_out = plan.t2_fit(sig, fa_out["fa_index"], out=t2_out)
    # ---- device-resident throughput (`value`)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    barrier()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
          for _ in range(args.steps)]
    l0 = lib.met2_launch_count()
    t_wall0 = time.time()
    for k in range(args.steps):
        ev[k][0].record()
        fa_out = plan.fa_fit(sig, out=fa_out)
        ev[k][1].record()
        t2_out = plan.t2_fit(sig, fa_out["fa_index"], out=t2_out)
        ev[k][2].record()
    barrier()
    t_wall1 = time.time()
    launches = lib.met2_launch_count() - l0
    total_ms = ev[0][0].elapsed_time(ev[-1][2])
    fa_ms = float(np.mean([e[0].elapsed_time(e[1]) for e in ev]))
    t2_ms = float(np.mean([e[1].elapsed_time(e[2]) for e in ev]))
    clocks = sampler.stop(t_wall0, t_wall1) if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, fa_out, t2_out)

    # ---- end to end through the public API with host buffers (H2D + fit + D2H inside the timed region)
    pinned = pipeline.host_buffers(plan, V)
    sig_np = sig_host.numpy()
    pipeline.fit_voxels(plan, sig_np, pinned_out=pinned)
    e2e_steps = max(1, min(args.steps, 3))
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(e2e_steps):
        res = pipeline.fit_voxels(plan, sig_np, pinned_out=pinned)
    e1.record()
    barrier()
    e2e_ms = e0.elapsed_time(e1) / e2e_steps
    h2d = int(sig_host.numel() * 8)
    d2h = int(sum(t.numel() * t.element_size() for t in pinned.values()))
    mwf_mean = float(res["maps"][:, 0].mean())

    # ---- ONE volume over the N GPUs of the node (north star: "a 96x96x60 brain in under 1 s on 8 B200")
    one = None
    if world > 1:
        one = one_volume(args, torch, dist, pipeline, plan, dev, rank, world, host_group, shape, barrier)

    t = torch.tensor([total_ms, e2e_ms, fa_ms, t2_ms], dtype=torch.float64, device=dev)
    lt = torch.tensor([launches], dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(lt, op=dist.ReduceOp.SUM)
    total_ms, e2e_ms, fa_ms, t2_ms = [float(x) for x in t.tolist()]
    launches = int(lt.item())
    if rank == 0:
        ms_per_step = total_ms / args.steps
        value = world * V / (ms_per_step * 1e-3)
        F = f_alg()
        rec = _ncu_record()
        hbm_peak, hbm_src = _hbm_peak()
        echo = not args.gram
        t2_kernel = "t2_echo_x2_kernel<1>" if echo else "t2_fit_kernel<2,1,X2>"

        def kernel_roofline(name, ms, falg, sd, bytes_per_voxel, key):
            ach = falg * V / (ms * 1e-3) / 1e12
            r = rec.get(key, {})
            ex = r.get("executed_fp64_flops_per_voxel")
            return {"kernel": name, "ms": ms, "achieved": ach, "peak": FP64_PEAK_TFLOPS, "unit": "TFLOP/s",
                    "frac_algorithmic": ach / FP64_PEAK_TFLOPS,
                    "algorithmic_flops_per_voxel": falg, "algorithmic_flops_per_voxel_sd": sd,
                    "executed_tflops": (ex * V / (ms * 1e-3) / 1e12) if ex else None,
                    "frac_executed": (ex * V / (ms * 1e-3) / 1e12 / FP64_PEAK_TFLOPS) if ex else None,
                    "traffic": (r.get("dram_bytes_per_voxel") * V) if r.get("dram_bytes_per_voxel") else None,
                    "algorithmic_bytes": bytes_per_voxel * V,
                    "hbm_achieved_gbs": bytes_per_voxel * V / (ms * 1e-3) / 1e9,
                    "from": (NCU_RECORD + ":" + key) if r else None}
        r_t2 = kernel_roofline(t2_kernel, t2_ms, F["F_alg_t2_x2_I"], F.get("F_alg_t2_x2_I_sd"), HBM_BYTES_PER_VOXEL_T2,
                               "t2_echo_x2" if echo else "t2_fit_x2")
        r_fa = kernel_roofline("fa_search_thread_kernel<32> + fa_search_kernel<2,1> (hand-backs) + fa_select_kernel<2,1>", fa_ms,
                               F["F_alg_fa_spline"],
                               F.get("F_alg_fa_spline_sd"), HBM_BYTES_PER_VOXEL_FA, "fa_spline")
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": n_warm, "warmup_requested": args.warmup, "ms_per_step": ms_per_step,
                "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": CONFIG,
                "run": {"t2_flags": args.t2_flags, "t2_kernel": t2_kernel, "voxels_per_gpu": V,
                        "l2": "inputs (142 MB) + outputs (0.44 GB) per step exceed the 126 MB L2; no explicit flush",
                        "stage_ms": {"fa": fa_ms, "t2": t2_ms}},
                "clocks": clocks,
                "e2e": {"value": world * V / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d,
                        "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms},
                "gpu_launches": launches,
                "roofline": dict(r_t2, bound="fp64", frac=r_t2["frac_algorithmic"],
                                 note="FP64 issue/latency bound, not HBM or tensor (SURVEY.md 8d). achieved = algorithmic "
                                      "flops of the REFERENCE formulation (Lawson-Hanson QR, cold starts; oracle/F_ALG.json, "
                                      "%d voxels) x voxels / kernel time (CUDA events): the reduced-echo-space, warm-started "
                                      "kernel needs far fewer, so frac_algorithmic can exceed 1; frac_executed = FP64 flops "
                                      "the kernel really issues (ncu counters of the committed capture named in `from`) / "
                                      "peak. peak = own DFMA microbench (MEASURED_PEAKS.json has no FP64 entry); HBM peak "
                                      "%.0f GB/s %s" % (F["n_voxels"], hbm_peak, hbm_src),
                                 hbm_peak_gbs=hbm_peak, kernels=[r_t2, r_fa]),
                "check": {"mwf_mean": mwf_mean}}
        if one is not None:
            line["one_volume"] = one
        if world == 1 and not args.no_cpu_baseline:
            os.environ.setdefault("OMP_NUM_THREADS", "1")
            cpu_setup()
            nvox, dt = cpu_run(CPU_SAMPLE_ROWS, seed=2)
            line["cpu_baseline"] = dict(cpu_env(), value=nvox / dt, unit=UNIT,
                                        sample="%d voxels (96x%dx1 slab of the config-2 phantom), %.1f s" % (
                                            nvox, CPU_SAMPLE_ROWS, dt))
            _CPU_STATE["pool"].close()
        if json_fd is None:
            print(json.dumps(line), flush=True)
        else:
            os.write(json_fd, (json.dumps(line) + "\n").encode())
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def dump_outputs(out_dir, fa_out, t2_out):
    """The arrays plan.fa_fit / plan.t2_fit returned in the last timed step, as <out_dir>/<name>.npy in float64 (the
    int32 outputs fa_index, fa_status and status convert exactly).  Per-voxel arrays are cut to the rows listed in
    voxel_index.npy: all voxels up to DUMP_VOXELS, else a sorted sample of DUMP_VOXELS drawn with seed 0."""
    import torch
    V = fa_out["fa_index"].shape[0]
    pick = np.arange(V) if V <= DUMP_VOXELS else np.sort(np.random.default_rng(0).choice(V, DUMP_VOXELS, replace=False))
    rows = torch.as_tensor(pick, device=fa_out["fa_index"].device)
    arrays = {"voxel_index": pick, "fsol_sum": fa_out["fsol_sum"].cpu().numpy()}
    for name, t in (("fa_index", fa_out["fa_index"]), ("fa_deg", fa_out["fa_deg"]), ("km", fa_out["km"]),
                    ("fa_status", fa_out["status"]), ("fsol", t2_out["fsol"]), ("est_signal", t2_out["est_signal"]),
                    ("reg", t2_out["reg"]), ("maps", t2_out["maps"]), ("status", t2_out["status"])):
        arrays[name] = t.index_select(0, rows).cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, dtype=np.float64))


def one_volume(args, torch, dist, pipeline, plan, dev, rank, world, host_group, shape, barrier):
    """ONE config-2 volume (seed 2) spread over the N GPUs, host memory in -> host memory out, two ways:
      (a) the product API: pipeline.MultiGpuFit in ONE process (what motor_recon_met2 does with num_cores = N): a host
          device copies its chunks of the pinned input, fits, and copies every output into its rows of one set
          of pinned host arrays.  Measured on rank 0 (wall clock around the call: it is a host API) while the other
          ranks wait on a HOST barrier, their GPUs idle;
      (b) one process per GPU (this torchrun job): every rank copies in its chunks, fits, and the outputs are gathered
          as slabs over NCCL (pipeline.gather_slabs is the same exchange) and read back on rank 0.  CUDA-event time,
          max over ranks.
    (a) is also timed with rank 0's GPU alone (same host-to-host path) for the strong-scaling efficiency of this run."""
    from multicomponent_t2_toolbox_b200.phantom import make_phantom
    steps = max(1, min(args.steps, 5))
    ph0 = make_phantom(shape, n_echoes=N_ECHOES, tau=TAU, TR=TR, seed=2, fa_mode="b1", backend="gpu")
    vol = torch.as_tensor(ph0["data"].reshape(-1, N_ECHOES)).pin_memory()
    V = vol.shape[0]
    out = {}
    # ---- (b) per-rank chunks + NCCL gather of slabs + D2H on rank 0
    deal = pipeline.chunk_deal(V, world)
    ranges = deal[rank]
    Vd = sum(hi - lo for lo, hi in ranges)
    nmax = max(sum(hi - lo for lo, hi in r) for r in deal)
    d_sig = torch.empty((nmax, N_ECHOES), dtype=torch.float64, device=dev)
    keys = ("fsol", "est_signal", "maps", "reg")
    widths = {"fsol": plan.npc, "est_signal": N_ECHOES, "maps": 6, "reg": 1}
    wtot = sum(widths.values()) + 3            # + fa_deg, km, (fa_index, status) packed into one float64
    slab = torch.zeros((nmax, wtot), dtype=torch.float64, device=dev)
    gathered = torch.empty((world * nmax, wtot), dtype=torch.float64, device=dev) if rank == 0 else None
    host_all = torch.empty((world * nmax, wtot), dtype=torch.float64).pin_memory() if rank == 0 else None

    def run_b():
        o = 0
        for lo, hi in ranges:
            d_sig[o:o + hi - lo].copy_(vol[lo:hi], non_blocking=True)
            o += hi - lo
        fa = plan.fa_fit(d_sig[:Vd])
        t2 = plan.t2_fit(d_sig[:Vd], fa["fa_index"])
        c = 0
        for k in keys:
            slab[:Vd, c:c + widths[k]] = t2[k].reshape(Vd, -1)
            c += widths[k]
        slab[:Vd, c] = fa["fa_deg"]
        slab[:Vd, c + 1] = fa["km"]
        slab[:Vd, c + 2] = fa["fa_index"].to(torch.float64) + 1024.0 * t2["status"].to(torch.float64)
        dist.gather(slab, list(gathered.split(nmax)) if rank == 0 else None, dst=0)
        if rank == 0:
            host_all.copy_(gathered, non_blocking=True)
    for _ in range(2):
        run_b()
    barrier()
    s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s0.record()
    for _ in range(steps):
        run_b()
    s1.record()
    barrier()
    tb = torch.tensor([s0.elapsed_time(s1) / steps], dtype=torch.float64, device=dev)
    dist.all_reduce(tb, op=dist.ReduceOp.MAX)
    out["per_rank_nccl_gather"] = {"ms": float(tb.item()), "h2d_bytes": int(V * N_ECHOES * 8),
                                   "gathered_bytes": int(world * nmax * wtot * 8),
                                   "note": "one process per GPU: H2D of its chunks, fit, dist.gather of slabs to rank 0 "
                                           "(NCCL), D2H on rank 0; CUDA events, max over ranks"}
    # ---- (a) the product API in one process on rank 0, the other ranks' GPUs idle (host barrier)
    if rank == 0:
        try:
            n_dev = torch.cuda.device_count()
            multi = pipeline.MultiGpuFit.create(min(world, n_dev), N_ECHOES, TAU, TR, reg_method=REG_METHOD,
                                                reg_matrix=REG_MATRIX, FA_method=FA_METHOD, t2_flags=args.t2_flags,
                                                echo_space=not args.gram)
            bufs = pipeline.host_buffers(plan, V)
            for _ in range(2):
                multi.fit(vol, out=bufs)
            t0 = time.perf_counter()
            for _ in range(steps):
                r = multi.fit(vol, out=bufs)
            a_ms = 1e3 * (time.perf_counter() - t0) / steps
            mwf_multi = float(r["maps"][:, 0].mean())
            single = pipeline.MultiGpuFit([plan])
            for _ in range(2):
                single.fit(vol, out=bufs)
            t0 = time.perf_counter()
            for _ in range(steps):
                r1 = single.fit(vol, out=bufs)
            single_ms = 1e3 * (time.perf_counter() - t0) / steps
            out["multi_gpu_fit"] = {"ms": a_ms, "gpus": len(multi.plans), "single_gpu_ms": single_ms,
                                    "strong_efficiency": single_ms / (len(multi.plans) * a_ms),
                                    "mwf_mean": mwf_multi, "mwf_mean_single": float(r1["maps"][:, 0].mean()),
                                    "h2d_bytes": int(V * N_ECHOES * 8),
                                    "d2h_bytes": int(sum(t.numel() * t.element_size() for t in bufs.values())),
                                    "note": "pipeline.MultiGpuFit (the path of motor_recon_met2 with num_cores = N): one "
                                            "process, all GPUs enqueued from one thread, pinned host in -> pinned host out, no "
                                            "collective; wall clock around the call, other ranks' GPUs idle"}
        except Exception as exc:   # never lose the headline line over the extra measurement
            out["multi_gpu_fit"] = {"error": repr(exc)[:300]}
    dist.barrier(group=host_group)
    out["voxels"] = int(V)
    out["gpus"] = world
    return out


def main():
    args = parse_args()
    if args.impl == "reference":
        return run_reference(args)
    if args.gpus > 1 and "WORLD_SIZE" not in os.environ:
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(args.gpus),
               "--master-addr", "127.0.0.1", "--master-port", "29533", os.path.abspath(__file__)] + sys.argv[1:]
        return subprocess.call(cmd)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
