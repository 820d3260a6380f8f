#!/usr/bin/env python
"""bench.py — MSCKF updates/s of the hot path (UpdaterMSCKF::update steps 2-6) on BASELINE.json's configurations.

    python bench.py [--config 2] --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K --warmup W        # the reference's CPU arithmetic (oracle port), rank 0

One step = one update over one feature batch. Default workload = config 2: a captured rpng_sim update (stereo, 20+1
clone poses, 400 MSCKF features, full online calibration, N = 194; tests/golden/rpng_sim_stereo20_f400.case.gz, made by
tests/golden/make_rpng_sim_cases.py from the host simulator with seeds 0). Other configs: 1 (rpng_sim mono/11/50),
3 (synthetic 4096-feature batch), 4 (4-camera, 31 clone poses, 800 features), 5 (TSQR+EKF microbench 8000 x 500).

Prints ONE JSON line (rank 0). `value` = updates/s with inputs resident in HBM (CUDA events on the engine's stream, L2
flushed between steps); `e2e` = updates/s through the C-ABI call with host buffers (H2D/D2H inside the timed call).
`--dump-outputs DIR` also writes the last timed step's results (per-feature status / points / chi², dx, posterior P) as
DIR/<name>.npy; the inputs are fixed (captured cases, seed-0 synthetic batches), so two builds can be compared file by file.
"""
from __future__ import annotations

import argparse
import json
import os
import re
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FP64_PEAK_TFLOPS = 37.1  # measured on this pool's B200s: DMMA m8n8k4 and DFMA both saturate at 64 FMA/clk/SM (tools/ubench/fp64_rate.cu,
#                          profiles/ubench_r02.txt); MEASURED_PEAKS.json carries no FP64 entry


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index=0):
        self.index = index
        self.proc = None
        self.path = None

    def start(self):
        try:
            self.path = tempfile.NamedTemporaryFile(delete=False, suffix=".csv").name
            q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
                 "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "50", "-i", str(self.index)],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if not self.proc:
            return out
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 9:
                    continue
                sm.append(float(f[1]))
                mx.append(float(f[2]))
                for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], f[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            out = {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm)}
        return out


# ---------------------------------------------------------------------------------------------------------------- workloads
class Workload:
    def __init__(self, name, data, frame, feats, opts, P, max_state=256, mode="msckf"):
        self.name, self.data, self.frame, self.feats, self.opts, self.P, self.max_state, self.mode = name, data, frame, feats, opts, P, max_state, mode
        self.n_feats = feats.n_feats if feats is not None else 0


def load_workload(config: int, compress: int, features: int | None = None) -> Workload:
    from open_vins_b200 import capi, sim, simrun
    if config in (1, 2) and features is None:
        path = simrun.CASE_CONFIG1 if config == 1 else simrun.CASE_CONFIG2
        frame, feats, opts, P = simrun.load_case(path)
        opts.compress = compress
        opts.col_order = capi.COLS_CANONICAL
        name = ("rpng_sim mono, max_clones=11 (12 clone poses), 50 MSCKF features/update" if config == 1 else
                "rpng_sim stereo, max_clones=20 (21 clone poses in the window), 400 MSCKF features/update") + \
            f", calib extrinsics+intrinsics+imu+dt on (N={P.shape[0]}), radtan 752x480, sigma_px=1, chi2_mult=1, FEJ on, GLOBAL_3D"
        return Workload(name, "rpng_sim", frame, feats, opts, P)
    if config == 5:
        H, res, P = sim.make_compress_case(m=8000, n=500, seed=0, structured=False)
        w = Workload("TSQR+EKFUpdate microbench: H 8000 x 500 dense i.i.d. N(0,1), P = A A'/500 + 1e-4 I, sigma^2 = 1, N = n = 500", "synthetic",
                     None, None, None, P, max_state=512, mode="dense")
        w.H, w.res = H, res
        return w
    if config == 4:
        c = sim.make_update_case(n_feats=features or 800, n_clones=31, n_cams=4, seed=0, calib_ext=True, calib_intr=True, calib_imu=True, calib_dt=True)
        name = f"rpng_sim-like 4 cameras, max_clones=30 (31 clone poses), {c.feats.n_feats} MSCKF features/update, full calibration (N={c.layout.N}; MSCKF part of config 4)"
        mx = 640
    else:  # 2 with an explicit feature count, or 3
        n = features or (4096 if config == 3 else 400)
        c = sim.make_update_case(n_feats=n, n_clones=21, n_cams=2, seed=0, calib_ext=True, calib_intr=True, calib_imu=True, calib_dt=True)
        name = f"synthetic rpng_sim-like stereo batch (config 3 sweep point), 21 clone poses, {n} MSCKF features/update, full calibration (N={c.layout.N})"
        mx = 256
    opts = capi.default_opts(do_calib_camera_pose=1, do_calib_camera_intrinsics=1, col_order=capi.COLS_CANONICAL, compress=compress)
    return Workload(name, "synthetic", c.frame, c.feats, opts, c.P, max_state=mx)


# ---------------------------------------------------------------------------------------------------------------- CPU arm
def pin_to_one_core():
    """The reference update is single-threaded; BASELINE.md §3: the CPU arm runs pinned (taskset -c 0 equivalent)."""
    try:
        old = os.sched_getaffinity(0)
        os.sched_setaffinity(0, {min(old)})
        return old
    except Exception:
        return None


def unpin(old):
    if old:
        try:
            os.sched_setaffinity(0, old)
        except Exception:
            pass


def cpu_updates(w: Workload, n_updates: int | None = None, warm: int = 1, budget_s: float = 20.0):
    """Updates of the oracle (CPU restatement of the reference's Eigen arithmetic) on the workload, one pinned thread.
    n_updates None: as many as fit in about budget_s seconds of CPU work (at least one; the first run doubles as the warm-up
    when a single update already takes seconds). Returns (updates/s from the median, last result, times)."""
    from oracle import ovo_py
    ovo_py.build()
    old = pin_to_one_core()
    try:
        times, r = [], None
        t = time.perf_counter()
        r = ovo_py.msckf_update(w.frame, w.feats, w.opts, w.P, dumps=False)
        t_first = time.perf_counter() - t
        if n_updates is None:
            n_updates = max(1, min(60, int(budget_s / max(t_first, 1e-3))))
        if t_first > 2.0 or warm == 0:
            times.append(t_first)  # seconds-long updates: cache warm-up is noise, every run counts
            n_updates -= 1
        for i in range(n_updates):
            t = time.perf_counter()
            r = ovo_py.msckf_update(w.frame, w.feats, w.opts, w.P, dumps=False)
            times.append(time.perf_counter() - t)
    finally:
        unpin(old)
    return 1.0 / float(np.median(times)), r, times


def cpu_context(w: Workload, r):
    """How much of the CPU time is the reference's algorithm rather than the hardware: the same stacked system compressed by
    LAPACK's blocked Householder QR (numpy, one thread) next to the reference's column-major Givens sweep."""
    try:
        from threadpoolctl import threadpool_limits
        from oracle import ovo_py
        rr = ovo_py.msckf_update(w.frame, w.feats, w.opts, w.P, dumps=True)
        H, res = rr.get("H_big"), rr.get("res_big")
        if H is None or H.shape[0] <= H.shape[1]:
            return None
        old = pin_to_one_core()
        try:
            with threadpool_limits(limits=1):
                t = time.perf_counter()
                np.linalg.qr(np.column_stack([H, res]), mode="r")
                t_qr = time.perf_counter() - t
        finally:
            unpin(old)
        return {"lapack_householder_qr_s": t_qr, "reference_givens_compress_s": float(rr["times"][2]),
                "note": "same stacked system, one thread: most of the CPU arm's time is the reference's stride-m Givens sweep, which a blocked "
                        "Householder QR would cut by this ratio; the GPU/CPU ratio reflects the reference's algorithm as much as the hardware"}
    except Exception as e:  # context only
        return {"error": str(e)[:200]}


def run_reference(args, rank):
    """--impl reference: the reference's own CPU implementation of the path. The reference cannot be built in this image
    (Eigen/OpenCV/Boost absent), so this is the oracle port, one pinned thread like the reference's estimator thread."""
    if rank != 0:
        return
    from open_vins_b200 import capi
    w = load_workload(args.config, capi.COMPRESS_HOUSEHOLDER_TSQR, args.features)
    if w.mode != "msckf":
        print(json.dumps({"impl": "reference", "unavailable": "config 5 is a kernel microbenchmark; the reference arm runs the update configs"}))
        return
    K = args.steps
    from oracle import ovo_py
    ovo_py.build()
    old = pin_to_one_core()
    try:
        for _ in range(min(args.warmup, 1)):
            ovo_py.msckf_update(w.frame, w.feats, w.opts, w.P, dumps=False)
        t0 = time.perf_counter()
        for _ in range(K):
            r = ovo_py.msckf_update(w.frame, w.feats, w.opts, w.P, dumps=False)
        dt = time.perf_counter() - t0
    finally:
        unpin(old)
    ups = K / dt
    line = {
        "impl": "reference", "metric": "msckf_updates_per_sec", "value": ups, "unit": "updates/s", "n_gpus": args.gpus, "steps": K,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / K, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f64", "data": w.data, "feats_per_sec": ups * w.n_feats,
        "config": {"workload": w.name, "features_in": int(w.n_feats), "features_used": int(r["stats"].n_feats_used), "rows_stacked": int(r["stats"].rows_stacked),
                   "cols_stacked": int(r["stats"].cols_stacked), "state_dim": int(w.P.shape[0])},
        "cpu_baseline": {"value": ups, "unit": "updates/s", "cores": 1, "kind": "port",
                         "sample": f"{K} full updates of the {w.n_feats}-feature batch, one pinned thread (the reference update is single-threaded)"},
        "e2e": {"value": ups, "unit": "updates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "features_used": int(r["stats"].n_feats_used), "rows_stacked": int(r["stats"].rows_stacked), "cols_stacked": int(r["stats"].cols_stacked),
        "stage_s": {k: float(v) for k, v in zip(["triangulate", "create_system", "compress", "update"], r["times"])},
    }
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, update_outputs(r["out"], r["dx"], r["P"]))
    print(json.dumps(line), flush=True)


_SAVED_STDOUT = None


def quiet_stdout():
    """N>1: NCCL prints its version banner on stdout at communicator creation. The contract is ONE JSON line on stdout,
    so file descriptor 1 is pointed at stderr until the line is emitted."""
    global _SAVED_STDOUT
    if _SAVED_STDOUT is None:
        sys.stdout.flush()
        _SAVED_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line: dict):
    global _SAVED_STDOUT
    sys.stdout.flush()
    if _SAVED_STDOUT is not None:
        os.dup2(_SAVED_STDOUT, 1)
        os.close(_SAVED_STDOUT)
        _SAVED_STDOUT = None
    print(json.dumps(line), flush=True)


DUMP_LIMIT_BYTES = 64 << 20


def update_outputs(out, dx, P) -> dict:
    """The arrays an MSCKF update hands its caller: the per-feature results, the state correction and the posterior covariance.
    The C ABI leaves NaN where a rejected feature never got a value (no point after a failed triangulation, no chi² before the
    gate); its status says so, and 0 stands there instead. A non-finite value of a feature the update used is an error."""
    from open_vins_b200 import capi
    used = out.status == capi.FEAT_OK
    arrays = dict(status=out.status, anchor_cam=out.anchor_cam, anchor_clone=out.anchor_clone, dx=dx, P=P)
    for k in ("p_FinA", "p_FinG", "chi2"):
        a = getattr(out, k)
        bad = ~np.isfinite(a)
        if (bad.reshape(len(a), -1).any(axis=1) & used).any():
            raise SystemExit(f"bench.py: --dump-outputs: non-finite {k} of a feature the update used")
        arrays[k] = np.where(bad, 0.0, a)
    return arrays


def dump_outputs(path: str, arrays: dict):
    """--dump-outputs: DIR/<name>.npy per array, all float64 (status codes and indices are exact in it) and finite, so that two
    builds run with the same arguments can be compared output for output."""
    arrays = {k: np.asarray(v, dtype=np.float64) for k, v in arrays.items()}
    bad = [k for k, a in arrays.items() if not np.isfinite(a).all()]
    if bad:
        raise SystemExit(f"bench.py: --dump-outputs: non-finite values in {', '.join(bad)}")
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit(f"bench.py: --dump-outputs: {total} bytes of outputs exceed the {DUMP_LIMIT_BYTES >> 20} MiB limit")
    os.makedirs(path, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(path, k + ".npy"), a)


# ---------------------------------------------------------------------------------------------------------------- rooflines
def short_name(mangled: str) -> str:
    for k in ("k_feature_system", "k_triangulate", "k_cam_poses", "k_column_map", "k_cq_gram", "k_cq_reduce", "k_cq_chol_gram", "k_cq_chol_ekf",
              "k_cq_trsm", "k_cq_trmm", "k_take_z", "k_ekf_prep", "k_ekf_gemm1", "k_ekf_gemm", "k_ekf_downdate1", "k_ekf_downdate", "k_ekf_chol",
              "k_ekf_trsm", "k_tsqr_level", "k_tsqr_assemble", "k_gram"):
        if k in mangled:
            return k
    m = re.search(r"k_[a-z0-9_]+", mangled)  # any other kernel of the library: the identifier inside the mangled name
    return m.group(0) if m else mangled[:40]


def kernel_table(eng, w: Workload, repeats=5):
    """Per-kernel durations (us, median over `repeats` profiled updates) of the update pipeline, launch order aggregated by kernel."""
    eng.set_profile(True)
    acc = {}
    order = []
    for _ in range(repeats):
        eng.cov_set(w.P)
        eng.msckf_update(w.frame, w.feats, w.opts)
        per = {}
        for nm, us in eng.profile_read():
            s = short_name(nm)
            per.setdefault(s, []).append(us)
            if s not in order:
                order.append(s)
        for s, v in per.items():
            acc.setdefault(s, []).append((len(v), float(np.sum(v))))
    eng.set_profile(False)
    return [{"kernel": s, "launches": acc[s][0][0], "us_per_step": float(np.median([t for _, t in acc[s]]))} for s in order]


def ncu_traffic(kernel: str):
    """dram bytes (read + write) per launch of `kernel` from the committed ncu --set full summary of this round, or None."""
    p = os.path.join(ROOT, "profiles", "ncu_r02_summary.json")
    try:
        d = json.load(open(p))
        k = d["kernels"][kernel]
        return float(k["dram_bytes_read"] + k["dram_bytes_write"]), f"profiles/ncu_r02_summary.json ({d.get('how', 'ncu --set full, cold cache')})"
    except Exception:
        return None, None


def rooflines(w: Workload, stats, stage_ms, ktab, nt_cols):
    """Roofline entries: the dominant kernel first (contract key `roofline`), then one entry per remaining heavy kernel."""
    hbm_peak, peak_src = peaks()
    m, n = int(stats.rows_stacked), int(stats.cols_stacked)
    kt = {k["kernel"]: k for k in ktab}
    M = w.feats.meas_off[1:] - w.feats.meas_off[:-1]
    m_all = int(np.maximum(2 * M - 3, 0).sum())  # rows of the staged system incl. the (zero) rows of rejected features
    out = []
    # per-feature kernel: writes the stacked rows once -> HBM-write bound in principle
    if "k_feature_system" in kt:
        t = stage_ms[1] * 1e-3  # the size classes run concurrently on three streams: the stage time IS the kernel group's duration
        by = 8.0 * m_all * (nt_cols) + 20.0 * int(M.sum())
        tr, src = ncu_traffic("k_feature_system")
        out.append({"kernel": "k_feature_system (Jacobians + nullspace projection + chi2 gate, one CTA per feature; 3 size-class launches side by side)",
                    "bound": "hbm", "achieved": by / t / 1e9, "peak": hbm_peak, "unit": "GB/s", "frac": by / t / 1e9 / hbm_peak, "traffic": tr,
                    "traffic_source": src, "peak_source": peak_src, "launches_per_step": kt["k_feature_system"]["launches"],
                    "avg_launch_us": 1e6 * t, "algorithmic_bytes_per_launch": by,
                    "note": "algorithmic bytes = 8 B x staged rows x (n+1) written + 20 B/measurement read; the stage is bound by the latency of the longest "
                            "tracks' CTAs (chi2 Cholesky pivot chain, sparse S accumulation), not by HBM"})
    def fp64(kname, label, flops, extra=""):
        if kname not in kt:
            return
        t = kt[kname]["us_per_step"] * 1e-6
        tr, src = ncu_traffic(kname)
        out.append({"kernel": label, "bound": "tensor", "achieved": flops / t / 1e12, "peak": FP64_PEAK_TFLOPS, "unit": "TFLOP/s",
                    "frac": flops / t / 1e12 / FP64_PEAK_TFLOPS, "traffic": tr, "traffic_source": src,
                    "peak_source": "FP64 DMMA/DFMA rate measured with tools/ubench/fp64_rate.cu on this pool (no FP64 entry in MEASURED_PEAKS.json)",
                    "launches_per_step": kt[kname]["launches"], "avg_launch_us": 1e6 * t / kt[kname]["launches"], "flops_per_step": flops, "note": extra})
    nT = (nt_cols + 31) // 32
    fp64("k_cq_gram", "k_cq_gram (Gram matrix of the stacked system on the FP64 tensor pipe, DMMA m8n8k4; two passes)",
         2 * 2.0 * m_all * (nT * (nT + 1) // 2) * 1024, "flops = 2 passes x 2 x rows x upper 32x32 tiles x 1024")
    fp64("k_cq_trsm", "k_cq_trsm (A <- A R^-1 in registers, DMMA pushes + per-row substitution; stacked system once, EKF gain once)",
         1.0 * (m_all + w.P.shape[0]) * nt_cols * nt_cols, "flops = rows x n^2 (triangular solve)")
    fp64("k_cq_chol_gram", "k_cq_chol_gram (single-CTA DMMA Cholesky, 155 x 155, two passes)", 2 * nt_cols**3 / 3.0,
         "latency-bound by the 155-pivot chain (about 125 cycles per pivot), not by the pipe")
    return out


# ---------------------------------------------------------------------------------------------------------------- main legs
def bench_update(args, w: Workload, local_rank=0, dist=None, rank=0, world=1):
    """N = 1 method (also used on every rank when the update is replicated at N > 1): e2e through the C ABI with host buffers,
    then `value` as the device-resident replay with L2 flush, per-step CUDA events."""
    import torch
    from open_vins_b200 import capi
    F = w.n_feats
    eng = capi.Engine(max_state=w.max_state, max_feats=max(1024, F), max_meas=max(65536, int(w.feats.n_meas) + 1024), device=local_rank)
    eng.set_replay(True)
    K, W = args.steps, args.warmup

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
    sampler = ClockSampler(local_rank)
    for _ in range(W):
        eng.cov_set(w.P)
        st, out, dx, stats = eng.msckf_update(w.frame, w.feats, w.opts)
    barrier()
    if rank == 0:
        sampler.start()
    t_e2e = 0.0
    host_us = np.zeros(4)
    out_buf = capi.FeatOut(F)  # result arrays owned by the caller, reused across calls like a host filter would
    dx_buf = np.zeros(w.P.shape[0])
    for _ in range(K):
        eng.cov_set(w.P)
        torch.cuda.synchronize()
        t = time.perf_counter()
        st, out, dx, stats = eng.msckf_update(w.frame, w.feats, w.opts, out_buf, dx_buf)
        t_e2e += time.perf_counter() - t
        h = eng.last_host_us()
        host_us += [h["marshal_h2d_enqueue"], h["kernel_enqueue"], h["wait"], h["unpack"]]
    cnt = eng.last_counters()
    cnt["host_us"] = host_us / K
    barrier()
    ms, stage_sum = eng.msckf_replay(W + K, flush_l2=True)
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    # what a caller receives from the last timed step: the per-feature results and dx of the last C-ABI call, and the
    # posterior covariance the last device-resident replay left on the GPU (same prior and inputs as that call)
    outputs = update_outputs(out, dx, eng.cov_get()) if args.dump_outputs else None
    ms = ms[W:]
    t_dev = float(ms.sum()) * 1e-3
    stage_ms = stage_sum / float(W + K)
    if dist is not None:
        tt = torch.tensor([t_e2e, t_dev], dtype=torch.float64, device=torch.device("cuda", local_rank))
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        t_e2e, t_dev = float(tt[0]), float(tt[1])
    return dict(eng=eng, K=K, W=W, t_e2e=t_e2e, t_dev=t_dev, stage_ms=stage_ms, stats=stats, out=out, cnt=cnt, clocks=clocks, ms=ms,
                outputs=outputs)


def bench_dense(args, w: Workload, local_rank=0):
    """Config 5: compress (8000 x 500) + EKFUpdate through the staged entry points. H2D of the dense H is inside every call, so
    this is an e2e-style number; the device part is reported from the engine's CUDA-event total."""
    import torch
    from open_vins_b200 import capi
    eng = capi.Engine(max_state=512, max_feats=64, max_meas=4096, max_rows=8192, device=local_rank)
    K, W = args.steps, args.warmup
    n = w.H.shape[1]
    for _ in range(W):
        eng.cov_set(w.P)
        eng.ekf_update([0], [n], w.H, w.res, sigma2=1.0)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(K):
        eng.cov_set(w.P)
        _, dx = eng.ekf_update([0], [n], w.H, w.res, sigma2=1.0)
    dt = (time.perf_counter() - t0) / K
    outputs = dict(dx=dx, P=eng.cov_get()) if args.dump_outputs else None
    eng.set_profile(True)
    sums, prof = [], None
    for _ in range(5):
        eng.cov_set(w.P)
        eng.ekf_update([0], [n], w.H, w.res, sigma2=1.0)
        prof = eng.profile_read()
        sums.append(sum(us for _, us in prof))
    eng.set_profile(False)
    eng.close()
    return dt, K, W, prof, float(np.median(sums)) * 1e-6, outputs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=[1, 2, 3, 4, 5])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--compress", default="cholqr2", choices=["tsqr", "gram", "cholqr2"],
                    help="measurement compression: cholqr2 (default, csrc/k_cholqr.cu), tsqr (Householder), gram (one-pass normal equations)")
    ap.add_argument("--features", type=int, default=None, help="synthetic batch with this many features instead of the config's captured case")
    ap.add_argument("--no-sweep", action="store_true", help="N>1: skip the 4096-feature sharded sweep point")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last step returned to its caller as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank)
        return

    import torch
    import torch.distributed as dist
    from open_vins_b200 import capi, multigpu

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the engine has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        quiet_stdout()
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    compress = {"tsqr": capi.COMPRESS_HOUSEHOLDER_TSQR, "gram": capi.COMPRESS_NORMAL_EQUATIONS, "cholqr2": capi.COMPRESS_CHOLQR2}[args.compress]
    w = load_workload(args.config, compress, args.features)
    hbm_peak, peak_src = peaks()

    if w.mode == "dense":
        if rank == 0:
            dt, K, W, prof, t_kernels, outputs = bench_dense(args, w, local_rank)
            m, n = w.H.shape
            flops = 2.0 * m * n * n - (2.0 / 3.0) * n**3 + 4.0 * m * n + 2.0 * n * n * n + 2 * n**3 / 3.0 + 3.0 * n**3
            ktab = {}
            for nm, us in prof:
                s = short_name(nm)
                ktab.setdefault(s, [0, 0.0])
                ktab[s][0] += 1
                ktab[s][1] += us
            dom = max(ktab.items(), key=lambda kv: kv[1][1])
            t_dom = dom[1][1] * 1e-6
            by = 8.0 * m * (n + 1) + 4.0 * n * (n + 1)
            line = {"metric": "tsqr_ekf_updates_per_sec", "value": 1.0 / t_kernels, "unit": "updates/s", "n_gpus": 1, "steps": K, "warmup": W,
                    "ms_per_step": 1e3 * t_kernels, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                    "config": {"workload": w.name, "compress": "cholqr2 (blocked variant: 501 columns)",
                               "timing": "value = 1 / (sum of the CUDA-event durations of the update's kernels, H already on the device; median of 5); "
                                         "e2e = host clock around ovb_ekf_update incl. the 32 MB H2D of H"},
                    "e2e": {"value": 1.0 / dt, "unit": "updates/s", "ms_per_step": 1e3 * dt, "h2d_bytes_per_step": int(8 * m * (n + 2) + 8 * n * n),
                            "d2h_bytes_per_step": int(8 * n), "timing": "host clock around ovb_cov_set + ovb_ekf_update (H2D + compress + EKF + D2H)"},
                    "gpu_launches": int(sum(v[0] for v in ktab.values())) * K,
                    "kernels_us": {k: {"launches": v[0], "us": v[1]} for k, v in ktab.items()},
                    "roofline": {"kernel": dom[0] + " (dominant kernel of the 8000 x 500 compression + update)", "bound": "tensor",
                                 "achieved": flops / t_kernels / 1e12, "peak": FP64_PEAK_TFLOPS, "unit": "TFLOP/s", "frac": flops / t_kernels / 1e12 / FP64_PEAK_TFLOPS,
                                 "traffic": None, "peak_source": "FP64 DMMA/DFMA rate measured with tools/ubench/fp64_rate.cu on this pool",
                                 "hbm": {"one_pass_bytes": by, "achieved_gbs_dominant_kernel": by / t_dom / 1e9, "peak_gbs": hbm_peak, "peak_source": peak_src},
                                 "note": "whole update (compression + EKF) flops over the summed kernel time; at AI = n/4 flop/B the QR is FP64-bound, "
                                         "not HBM-bound; the dominant kernel's share is in kernels_us"}}
            if not args.no_cpu_baseline:
                from oracle import ovo_py
                ovo_py.build()
                old = pin_to_one_core()
                try:
                    ts = []
                    for _ in range(3):
                        t = time.perf_counter()
                        Rc, zc = ovo_py.compress(w.H, w.res)
                        ovo_py.ekf_update(w.P, [0], [n], Rc, zc, sigma2=1.0)
                        ts.append(time.perf_counter() - t)
                finally:
                    unpin(old)
                line["cpu_baseline"] = {"value": 1.0 / float(np.median(ts)), "unit": "updates/s", "cores": 1, "kind": "port",
                                        "sample": f"3 full 8000 x 500 compress + EKFUpdate runs of the oracle (median, {sum(ts):.1f} s), one pinned thread"}
            if outputs is not None:
                dump_outputs(args.dump_outputs, outputs)
            emit(line)
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    F = w.n_feats
    rows_total = multigpu.stacked_rows(w.feats.meas_off)
    replicated = world > 1 and rows_total < multigpu.REPLICATE_BELOW_ROWS
    if args.dump_outputs and world > 1 and not replicated:
        raise SystemExit("bench.py: --dump-outputs covers the single-GPU and replicated updates, not the sharded one")
    line = None
    if world == 1 or replicated:
        r = bench_update(args, w, local_rank, dist if world > 1 else None, rank, world)
        eng, K, W, stats = r["eng"], r["K"], r["W"], r["stats"]
        if rank == 0:
            value = K / r["t_dev"]
            m_rows, n_cols = int(stats.rows_stacked), int(stats.cols_stacked)
            ktab = kernel_table(eng, w)
            rl = rooflines(w, stats, r["stage_ms"], ktab, n_cols + 1)
            line = {
                "metric": "msckf_updates_per_sec", "value": value, "unit": "updates/s", "n_gpus": world, "steps": K, "warmup": W,
                "ms_per_step": 1e3 * r["t_dev"] / K, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": w.data,
                "feats_per_sec": value * F,
                "config": {"workload": w.name, "features_in": F, "features_used": int(stats.n_feats_used), "rows_stacked": m_rows, "cols_stacked": n_cols,
                           "state_dim": int(w.P.shape[0]), "l2": "flushed between steps (256 MiB memset)", "col_order": "canonical", "compress": args.compress,
                           "multi_gpu": (f"replicated on {world} ranks: {rows_total} stacked rows < {multigpu.REPLICATE_BELOW_ROWS}, sharding a sub-millisecond "
                                         "update only adds an all-gather and a second compression; every rank runs the whole update, no collective")
                           if replicated else "single GPU"},
                "e2e": {"value": K / r["t_e2e"], "unit": "updates/s", "ms_per_step": 1e3 * r["t_e2e"] / K, "h2d_bytes_per_step": r["cnt"]["h2d_bytes"],
                        "d2h_bytes_per_step": r["cnt"]["d2h_bytes"], "feats_per_sec": F * K / r["t_e2e"],
                        "timing": "host clock around the synchronous C-ABI call (marshalling + H2D + kernels + D2H), summed over steps"
                                  + (", max over ranks" if world > 1 else ""),
                        "host_us_inside_call": {k: float(v) for k, v in zip(["marshal_and_h2d_enqueue", "kernel_enqueue", "wait_for_stream", "unpack_results"],
                                                                           r["cnt"]["host_us"])}},
                "gpu_launches": r["cnt"]["launches"] * K, "gpu_launches_per_step": r["cnt"]["launches"],
                "stage_ms": {k: float(v) for k, v in zip(["triangulate", "feature_systems", "column_map", "compress", "ekf_update"], r["stage_ms"])},
                "step_ms_quantiles": {q: float(np.quantile(r["ms"], float(q))) for q in ("0.5", "0.9", "0.99")},
                "kernels_us": ktab,
                "roofline": rl[0] if rl else None, "rooflines": rl[1:],
                "clocks": r["clocks"],
            }
    else:
        # sharded: features over ranks, ONE all-gather of the compressed blocks per update
        cap = max(1024, F)
        eng = capi.Engine(max_state=w.max_state, max_feats=cap, max_meas=cap * 64, device=local_rank)
        be = multigpu.EngineBackend(eng, torch.device("cuda", local_rank))
        sampler = ClockSampler(local_rank)
        if rank == 0:
            sampler.start()
        K, W = args.steps, args.warmup
        r = multigpu.time_sharded(eng, be, dist, torch, w, w.opts, rank, world, K, W, 0)
        clocks = sampler.stop() if rank == 0 else None
        cnt = eng.last_counters()
        if rank == 0:
            line = {
                "metric": "msckf_updates_per_sec", "value": K / r["t_dev"], "unit": "updates/s", "n_gpus": world, "steps": K, "warmup": W,
                "ms_per_step": 1e3 * r["t_dev"] / K, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": w.data,
                "feats_per_sec": F * K / r["t_dev"],
                "config": {"workload": w.name, "features_in": F, "features_used": r["features_used"], "state_dim": int(w.P.shape[0]),
                           "multi_gpu": f"features sharded over {world} ranks, one NCCL all-gather of the compressed (R,z) block per update, EKF update replicated",
                           "l2": "inputs re-uploaded every step", "replicas_bitwise_equal": r["replicas_bitwise_equal"],
                           "sharded_vs_single_relerr": r["sharded_vs_single_relerr"], "gate_decisions_equal": r["gate_decisions_equal_on_all_ranks"]},
                "e2e": {"value": K / r["t_host"], "unit": "updates/s", "ms_per_step": 1e3 * r["t_host"] / K, "h2d_bytes_per_step": cnt["h2d_bytes"],
                        "d2h_bytes_per_step": cnt["d2h_bytes"], "timing": "host clock around shard_compress + all_gather + finish, max over ranks"},
                "gpu_launches": cnt["launches"] * K, "gpu_launches_per_step": cnt["launches"], "clocks": clocks,
                "roofline": {"bound": "hbm", "achieved": None, "peak": hbm_peak, "unit": "GB/s", "frac": None, "traffic": None,
                             "note": "per-rank kernels are those of the N=1 line"},
            }
    # ---- N > 1: the batch size at which sharding pays, in the same line (config-3 sweep point, 4096 features)
    if world > 1 and not args.no_sweep and args.config == 2:
        w3 = load_workload(3, compress, 4096)
        eng3 = capi.Engine(max_state=w3.max_state, max_feats=4096, max_meas=4096 * 64, device=local_rank)
        be3 = multigpu.EngineBackend(eng3, torch.device("cuda", local_rank))
        K3 = max(10, min(args.steps, 40))
        r3 = multigpu.time_sharded(eng3, be3, dist, torch, w3, w3.opts, rank, world, K3, 3, 0)
        # single-GPU time of the same batch on this rank, same event bracket (inputs resident -> EKF done)
        eng3.set_stream(be3.stream.cuda_stream)
        t1 = 0.0
        for i in range(3 + K3):
            eng3.cov_set(w3.P)
            with be3.stream_ctx():
                eng3.msckf_update(w3.frame, w3.feats, w3.opts)
            if i >= 3:
                t1 += float(np.sum(eng3.last_stage_ms()[:5])) * 1e-3
        tt = torch.tensor([t1], dtype=torch.float64, device=torch.device("cuda", local_rank))
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        if rank == 0 and line is not None:
            line["sweep_4096"] = {"workload": w3.name, "sharded_updates_per_sec": K3 / r3["t_dev"], "single_gpu_updates_per_sec": K3 / float(tt[0]),
                                  "speedup_vs_one_gpu": float(tt[0]) / r3["t_dev"], "e2e_updates_per_sec": K3 / r3["t_host"], "steps": K3,
                                  "replicas_bitwise_equal": r3["replicas_bitwise_equal"], "sharded_vs_single_relerr": r3["sharded_vs_single_relerr"],
                                  "timing": "CUDA events on the engine stream, inputs resident -> EKF update done, max over ranks"}
        eng3.close()
    if rank == 0 and line is not None:
        if not args.no_cpu_baseline and w.mode == "msckf":
            ups, rr, times = cpu_updates(w)
            n_cpu = len(times)
            if world == 1 or replicated:
                assert np.array_equal(rr["out"].status, r["out"].status), "GPU and CPU gate decisions differ on the bench workload"
            line["cpu_baseline"] = {"value": ups, "unit": "updates/s", "cores": 1, "kind": "port",
                                    "sample": f"{n_cpu} full updates of the same {F}-feature batch (median, {sum(times):.1f} s), one pinned thread; "
                                              f"{os.cpu_count()} logical cores on the box",
                                    "stage_s": {k: float(v) for k, v in zip(["triangulate", "create_system", "compress", "update"], rr["times"])},
                                    "context": cpu_context(w, rr)}
            line["speedup_e2e_vs_cpu_port"] = line["e2e"]["value"] / ups
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, r["outputs"])
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
