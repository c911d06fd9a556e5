#!/usr/bin/env python
"""bench.py — GH-ICP inner-loop benchmark (BASELINE.json metric: ICP iterations/s at N_src x N_tgt).

A "step" = one body of GHRegistration::ghicp_reg's while-loop (src/ghicp_reg.cpp:49-103, viewer
excluded): calED + calCD_* + findcorrespondence* + transformestimation + adjustweight.
Default workload = BASELINE.json configs[1]: 50k x 50k keypoints, BSC descriptors, KM matching, 6-DoF.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload ...] [--dump-outputs DIR]

Prints ONE JSON line (rank 0).  See DESIGN.md §Measurement for every field.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (N, M, feature, corr, bits)
    "config1": dict(N=2000, M=2000, ft="none", ct="nn", bits=0, desc="2k x 2k, no feature, NN, 6-DoF"),
    "config2": dict(N=50000, M=50000, ft="bsc", ct="km", bits=441, desc="50k x 50k, BSC-441 (reference's BSCEncoder(.,7)), KM, 6-DoF"),
    "config2-672": dict(N=50000, M=50000, ft="bsc", ct="km", bits=672, desc="50k x 50k, BSC-672, KM, 6-DoF"),
    "config2-nn": dict(N=50000, M=50000, ft="bsc", ct="nn", bits=441, desc="50k x 50k, BSC-441, NN, 6-DoF"),
    "config2-nnr": dict(N=50000, M=50000, ft="bsc", ct="nnr", bits=441, desc="50k x 50k, BSC-441, NNR, 6-DoF"),
    # BASELINE.json configs[2]: no N x M array fits (reference: 320 GB of doubles; stored float plane: 160 GB) ->
    # matrix-free FPFH path (gh-icp_b200/csrc/ghicp_fpfh.cu); point-to-point solve like the reference loop
    "config3": dict(N=200000, M=200000, ft="fpfh", ct="nnr", bits=0, desc="200k x 200k, FPFH-33 float, NN + reciprocal, matrix-free"),
    # BASELINE.json configs[3] / [4]: RAW scans -> voxel filter + curvature keypoints + BSC encoder on the GPU (device-resident
    # pipeline, ghicp_prep_run) -> KM registration of the keypoint sets (N, M = what the detector finds; filled in at run time)
    "config4": dict(N=0, M=0, raw=1000000, overlap=0.6, dof=6, ft="bsc", ct="km", bits=441, voxel=0.05, radius=0.5, nms=1.0,
                    desc="1M + 1M raw points -> voxel 0.05 m + curvature keypoints + BSC-441 on the GPU -> KM, 6-DoF"),
    "config5": dict(N=0, M=0, raw=5000000, overlap=0.3, dof=4, ft="bsc", ct="km", bits=441, voxel=0.05, radius=0.5, nms=1.0,
                    desc="5M + 5M raw points, 30 % overlap -> voxel 0.05 m + keypoints + BSC-441 (2 variants: '4-DoF leveled') -> KM"),
}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region (NVML, every 10 ms; nvidia-smi fallback)."""

    def __init__(self, dev=0):
        self.rows, self.stop, self.dev = [], threading.Event(), dev
        self.t = None
        self.nv = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(dev)
        except Exception:
            self.nv = None

    def _run(self):
        nv = self.nv
        while not self.stop.is_set():
            try:
                if nv is not None:
                    sm = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                    mx = nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM)
                    rs = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                        else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                    self.rows.append((sm, mx, rs))
                    self.stop.wait(0.01)
                else:
                    q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
                         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
                    out = subprocess.run(["nvidia-smi", f"--id={self.dev}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                         capture_output=True, text=True, timeout=5).stdout
                    r = [x.strip() for x in out.strip().split(",")]
                    bits = 0
                    for k, v in enumerate(r[2:6]):
                        if v.lower().startswith("active"):
                            bits |= [0x8, 0x40, 0x20, 0x4][k]
                    self.rows.append((float(r[0]), float(r[1]), bits))
                    self.stop.wait(0.1)
            except Exception:
                self.stop.wait(0.05)

    def __enter__(self):
        self.t = threading.Thread(target=self._run, daemon=True)
        self.t.start()
        return self

    def __exit__(self, *a):
        self.stop.set()
        self.t.join(timeout=6)

    def summary(self):
        sm = [r[0] for r in self.rows]
        mx = max([r[1] for r in self.rows], default=0)
        bits = 0
        for r in self.rows:
            bits |= int(r[2])
        names = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}
        reasons = sorted(n for b, n in names.items() if bits & b)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": float(mx) or None,
                "reasons": reasons, "samples": len(sm)}


_RAW_CACHE = {}


def raw_scans(g, wl):
    key = (wl["raw"], wl["overlap"])
    if key not in _RAW_CACHE:
        _RAW_CACHE[key] = g.synth.scan_pair(wl["raw"], wl["overlap"], seed=4)
    return _RAW_CACHE[key]


def make_scene_from_raw_cpu(g, wl, raw_points):
    """CPU arm of the pipeline workloads: the ORACLE's voxel filter + keypoint detector + BSC encoder (test infrastructure, the
    restated include/filter.hpp, keypoint_detect.hpp, pca.h, binary_feature_extraction.hpp) on a crop of the raw scans
    (a band in y, which keeps the overlap ratio along x) of about `raw_points` points each."""
    import oracle
    Tc, Sc, _, _ = raw_scans(g, wl)
    frac = min(1.0, raw_points / float(wl["raw"]))
    pat = g.bsc_default_pattern(7)
    out, t_prep = {}, time.perf_counter()
    for name, P, dof in (("T", Tc, 0), ("S", Sc, wl["dof"])):
        if frac < 1.0:
            y = P[:, 1]
            P = np.ascontiguousarray(P[y < np.quantile(y, frac)])
        D = np.ascontiguousarray(P[oracle.voxel_downsample(P, wl["voxel"])])
        kp, _, _, _ = oracle.detect_keypoints(D, wl["radius"], 0.65, 20, wl["nms"])
        bits = oracle.bsc_extract(D, kp, wl["nms"], pat, 7, dof)[0]
        out[name] = (D, kp, bits)
    t_prep = time.perf_counter() - t_prep
    D, kp, _ = out["S"]
    ext = D.max(axis=0) - D.min(axis=0)
    sc = g.synth.Scene(S=np.asfortranarray(out["S"][0][out["S"][1]].astype(np.float64)),
                       T=np.asfortranarray(out["T"][0][out["T"][1]].astype(np.float64)),
                       bbx_magnitude=float(np.float32(ext[0] + ext[1] + ext[2])), R_gt=None, t_gt=None, n_overlap=0, perm=None)
    sc.bsc_s, sc.bsc_t, sc.bits = out["S"][2], out["T"][2][0], 441
    sc.meta = dict(cpu_prep_s=t_prep, raw_points=int(raw_points))
    return sc


def make_scene(g, wl, n_override=None, seed=2):
    if "raw" in wl:
        return make_scene_from_raw_cpu(g, wl, n_override or wl["raw"])
    N = n_override or wl["N"]
    M = n_override or wl["M"]
    if wl["ft"] == "none":
        sc = g.synth.gen_points(N, M, overlap=0.9, extent=(100, 100, 20), noise=0.02, seed=1)
    else:
        # same point density as config 2 at any size (so candidate statistics stay comparable)
        f = (N / 50000.0) ** (1.0 / 3.0)
        sc = g.synth.gen_points(N, M, overlap=0.6, extent=(200 * f, 200 * f, 40 * f), noise=0.05, seed=seed)
        if wl["ft"] == "bsc":
            g.synth.add_bsc(sc, bits=wl["bits"], V=4)
        elif wl["ft"] == "fpfh":
            g.synth.add_fpfh(sc)
    return sc


# dram__bytes_read.sum + dram__bytes_write.sum of ONE k_stream launch, from the committed `ncu --set full` captures
# (profiles/r01_summary.md); algorithmic bytes are 5.002e9
# dram__bytes_read.sum + dram__bytes_write.sum of the dominant kernel's launch in an `ncu --set full` capture of the same command
# (a constant from the committed capture, labelled with its source: a bench run is never taken under the profiler)
NCU_TRAFFIC = {"config2": {"bytes": 5.038999e9 + 0.32185856e9,
                           "source": "profiles/r02_ncu_k_stream_km.raw.csv (ncu --set full, k_stream<2,1,1,1,1>, round 2): "
                                     "5.039 GB read (algorithmic 5.002 GB) + 0.322 GB written (counts, partial sums, edge list)"},
               "config2-672": {"bytes": 5.038999e9 + 0.32185856e9,
                               "source": "profiles/r02_ncu_k_stream_km.raw.csv (the same kernel and plane: the descriptor width only "
                                         "changes the one-time FD build)"},
               "config2-nnr": {"bytes": 5.179896e9 + 0.321731584e9,
                               "source": "profiles/r02_ncu_k_stream_nnr.raw.csv (ncu --set full, k_stream<1,1,1,1,1>, round 2)"},
               "config2-nn": {"bytes": 5.311e9, "source": "profiles/r01_summary.md (ncu --set full capture of k_stream NN, round 1)"}}

DUMP_BYTES = 64 << 20   # --dump-outputs writes at most this much; a larger array is replaced by a seeded sample of its rows


def dump_outputs(out_dir, arrays):
    """Writes each array as out_dir/<name>.npy (float64), rows sampled with a fixed seed where the whole would not fit."""
    os.makedirs(out_dir, exist_ok=True)
    budget = DUMP_BYTES // len(arrays)
    for name, a in arrays.items():
        a = np.asarray(a, dtype=np.float64)
        if a.nbytes > budget:
            rows = budget // max(1, a.nbytes // max(1, len(a)))
            a = a[np.sort(np.random.default_rng(0).choice(len(a), rows, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a))


FT = {"none": 3, "bsc": 0, "fpfh": 2}
CT = {"nn": 0, "nnr": 1, "km": 2}


# --------------------------------------------------------------------------------------------------
# CPU arm: the REFERENCE's own loop (oracle/_ref/libghreg_ref.so = src/ghicp_reg.cpp + km.cpp + stereo_binary_feature.cpp
# compiled verbatim, one thread like the reference) or, where that build is absent, the oracle port.  Iteration-matched:
# the CPU times the SAME iteration indices the GPU arm times (warm-up iterations 0..W-1 are run, not timed; steps are
# iterations W..W+K-1), on a bounded n_s x n_s sample of the workload generated by the same make_scene().  The workload-size
# figure is an extrapolation t(N) = t(n_s) * (N / n_s)^p with p FITTED on >= 2 sample sizes (not assumed), and is labelled so.
# --------------------------------------------------------------------------------------------------
def _cpu_loop(g, wl, n, n_iters, kind, threads=1, stop_at_convergence=False):
    """Per-iteration wall ms of the CPU loop from iteration 0 on an n x n sample; returns (list ms, fd_build_s, converged_at)."""
    import oracle
    import tempfile
    sc = make_scene(g, wl, n_override=n)
    dof = wl.get("dof", 6)
    cwd = os.getcwd()
    os.chdir(tempfile.mkdtemp())  # Km::output writes Corres.txt (src/km.cpp:148)
    try:
        if kind == "reference":
            o = oracle.Reference(FT[wl["ft"]], CT[wl["ct"]], dof=dof, bbx_magnitude=sc.bbx_magnitude, solve_mode=0)
        else:
            o = oracle.Oracle(FT[wl["ft"]], CT[wl["ct"]], dof=dof, bbx_magnitude=sc.bbx_magnitude, solve_mode=0,
                              use_ref_km=(oracle.ref_km_lib() is not None and wl["ct"] == "km"), num_threads=threads)
        o.set_keypoints(sc.S, sc.T)
        if wl["ft"] == "bsc":
            o.set_bsc(sc.bsc_s, sc.bsc_t, sc.bits)
        elif wl["ft"] == "fpfh":
            o.set_fpfh(sc.fpfh_s, sc.fpfh_t)
        t0 = time.perf_counter()
        o.build_fd()
        t_fd = time.perf_counter() - t0
        ts, conv_at = [], None
        for it in range(n_iters):
            t0 = time.perf_counter()
            st = o.iterate()
            ts.append((time.perf_counter() - t0) * 1e3)
            if st.converged and conv_at is None:
                conv_at = it + 1
                if stop_at_convergence:
                    break
    finally:
        os.chdir(cwd)
    return ts, t_fd, conv_at, max(sc.S.shape[0], sc.T.shape[0]), dict(getattr(sc, "meta", {}) or {})


def _fit_power(ns, ts):
    """Least-squares exponent p and prefactor of t = a * n^p on log-log axes."""
    ln, lt = np.log(np.asarray(ns, float)), np.log(np.maximum(np.asarray(ts, float), 1e-9))
    if len(ns) < 2:
        return None, None
    p, la = np.polyfit(ln, lt, 1)
    return float(p), float(math.exp(la))


def cpu_arm(g, wl, warmup, steps, sizes, fit_steps=3, threads=1, budget_s=240.0):
    """Iteration-matched CPU measurement.  `sizes` ascending; the LAST size is the main sample: warm-up + `steps` timed
    iterations there; the smaller sizes run warm-up + `fit_steps` iterations and only feed the exponent fit."""
    import oracle
    oracle.build()
    kind = "reference" if (oracle.ref_ghreg_lib() is not None and threads == 1) else "port"
    raw = "raw" in wl                     # pipeline workloads: `sizes` are RAW points per scan, n = the keypoints they yield
    N = wl["N"]
    sizes = sorted(set(min(s, wl["raw"] if raw else N) for s in sizes))
    rows, t_start = [], time.perf_counter()
    for k, n_req in enumerate(sizes):
        main = (k == len(sizes) - 1)
        n_it = warmup + (steps if main else min(steps, fit_steps))
        ts, t_fd, conv_at, n, meta = _cpu_loop(g, wl, n_req, n_it, kind, threads)
        if raw and main and N <= 0:         # full keypoint count unknown on the CPU side: keypoints scale with the scanned area
            N = int(round(n * wl["raw"] / float(n_req)))
        timed = ts[warmup:]
        rows.append(dict(n=n, meta=meta, iteration_ms=[round(t, 3) for t in ts], timed_mean_ms=float(np.mean(timed)),
                         timed_median_ms=float(np.median(timed)), fd_build_s=t_fd, converged_at=conv_at,
                         registration_ms=float(np.sum(ts[:conv_at])) if conv_at else None))
        if time.perf_counter() - t_start > budget_s and not main:
            # out of time for the ladder: the next size is the main sample anyway
            continue
    main_row = rows[-1]
    n_s = main_row["n"]
    ms_sample = main_row["timed_mean_ms"]
    extrap = n_s < N
    p_steady, _ = _fit_power([r["n"] for r in rows], [r["timed_median_ms"] for r in rows])
    fit = None
    ms_full = ms_sample
    reg = None
    if extrap:
        if p_steady is None:   # a single sample size: the documented asymptotics (cost ~ N*M; KM ~ n^3)
            p_steady = 3.0 if wl["ct"] == "km" else 2.0
            fit_src = "assumed (single sample size)"
        else:
            fit_src = f"fitted on n = {[r['n'] for r in rows]}"
        ms_full = ms_sample * (N / n_s) ** p_steady
        fit = dict(exponent=p_steady, source=fit_src,
                   samples=[[r["n"], r["timed_median_ms"]] for r in rows])
    # whole registration (iteration 0 .. convergence): measured at the sample sizes, extrapolated with its own exponent
    regs = [(r["n"], r["registration_ms"]) for r in rows if r["registration_ms"]]
    if regs:
        p_reg, _ = _fit_power([a for a, _ in regs], [b for _, b in regs])
        n_r, ms_r = regs[-1]
        conv = [r["converged_at"] for r in rows if r["n"] == n_r][0]
        reg = dict(sample_n=n_r, iterations=conv, ms_total_sample=ms_r, ms_per_iteration_sample=ms_r / conv)
        if n_r < N:
            pr = p_reg if p_reg is not None else p_steady
            reg.update(extrapolated=True, exponent=pr, ms_per_iteration=ms_r / conv * (N / n_r) ** pr)
        else:
            reg.update(extrapolated=False, ms_per_iteration=ms_r / conv)
    what = ("the reference's own src/ghicp_reg.cpp + km.cpp + stereo_binary_feature.cpp compiled verbatim (oracle/_ref/"
            "libghreg_ref.so; 1 thread: it is single-threaded; PCL's SVD call delegated to the oracle)") if kind == "reference" \
        else f"oracle port of the reference loop ({threads} thread(s): OpenMP on the O(N*M) loops, KM serial)"
    sample = (f"{what}; iterations {warmup}..{warmup + steps - 1} of a registration from iteration 0 (the indices the GPU arm "
              f"times) on a {n_s}x{n_s} sample of the workload (same generator, same density"
              + ("; keypoints + descriptors from the oracle's pre-processing of a y-band of the raw scans" if raw else "")
              + f"): {ms_sample:.1f} ms/iteration"
              + (f"; extrapolated to {N} keypoints by (N/n_s)^{p_steady:.2f} ({fit['source']})" if extrap else "; no extrapolation"))
    return dict(value=1000.0 / ms_full, unit="iterations/s", cores=threads, kind=kind, sample=sample,
                ms_per_step_sample=ms_sample, sample_n=n_s, extrapolated=extrap, fit=fit, registration=reg, ladder=rows)


def main():
    # stdout carries exactly ONE JSON line: whatever libraries print on fd 1 while we run (NCCL's version banner, ...) goes to
    # stderr; the line itself is written to the saved descriptor at the end
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    try:
        _main(saved_stdout)
    finally:
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        os.close(saved_stdout)


def _main(saved_stdout):
    def emit(line):
        sys.stdout.flush()
        if sys.stdout is not sys.__stdout__:      # run in-process by a harness that replaced sys.stdout (pytest's capsys)
            print(json.dumps(line))
        else:
            os.write(saved_stdout, (json.dumps(line) + "\n").encode())

    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=4)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="config2", choices=sorted(WORKLOADS))
    ap.add_argument("--n", type=int, default=0, help="override N=M (e.g. 4000: a size the reference runs WITHOUT extrapolation)")
    ap.add_argument("--cpu-sample", type=int, default=0, help="N=M of the CPU arm's main sample")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned (pairs, keypoints, transforms, statistics) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.warmup < 3:
        args.warmup = 3  # timing rule: >= 3 warm-up steps

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    wl = dict(WORKLOADS[args.workload])
    if args.n:
        wl["N"] = wl["M"] = args.n
    import ghicp_b200 as g

    config = {"parallelism": f"source rows sharded over {args.gpus} GPU(s), target replicated" if args.gpus > 1 else "1 GPU",
              "workload": args.workload + (f" (N=M={args.n} override)" if args.n else ""), "desc": wl["desc"],
              "N_src": wl["N"], "N_tgt": wl["M"], "descriptor_bits": wl["bits"], "correspondence": wl["ct"],
              "timed_iterations": [args.warmup, args.warmup + args.steps - 1],
              "l2_policy": ("FD plane of the detected keypoint sets (tens of MB) stays L2-resident across iterations, as in a real "
                            "registration; no flush") if "raw" in wl else
              "inputs larger than L2 (FD plane u16 N x M streamed every step)" if wl["ft"] == "bsc"
              else "matrix-free; working set < L2 by construction"}
    ncores = os.cpu_count() or 1
    km = wl["ct"] == "km"

    # ---------------- reference arm: the reference's CPU implementation on the host cores ------------
    if args.impl == "reference":
        if rank != 0:
            return
        t0 = time.perf_counter()
        if "raw" in wl:
            cap = args.cpu_sample or 250000                # raw points per scan the oracle pre-processes on the CPU
            sizes = [min(wl["raw"], cap // 2), min(wl["raw"], cap)]
        elif wl["N"] <= 4000:
            sizes = [wl["N"]]                              # measured at the workload size, no extrapolation
        else:
            n_s = args.cpu_sample or (2000 if km else 6000)
            sizes = [max(500, n_s // 2), max(750, (3 * n_s) // 4), n_s]
        cb = cpu_arm(g, wl, args.warmup, args.steps, sizes, fit_steps=3)
        line = {"impl": "reference", "metric": "ICP iterations/sec", "value": cb["value"], "unit": "iterations/s",
                "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                # the time of one MEASURED step (an iteration of the bounded sample); `value` is the workload-size figure
                "ms_per_step": cb["ms_per_step_sample"], "ms_per_step_is": f"measured on the {cb['sample_n']}x{cb['sample_n']} sample",
                "value_is": "extrapolated to the workload size (see fit)" if cb["extrapolated"] else "measured at the workload size",
                "extrapolated": cb["extrapolated"], "fit": cb["fit"], "registration": cb["registration"],
                "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config,
                "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")},
                "e2e": {"value": cb["value"], "unit": "iterations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "ladder": cb["ladder"], "gpu_launches": 0, "wall_s": time.perf_counter() - t0}
        emit(line)
        return

    # ---------------- our arm --------------------------------------------------------------------------
    if g.device_count() <= 0:
        raise SystemExit("bench.py: no CUDA device (the product has no CPU fallback)")
    dist = None
    if world > 1:
        # stdout carries exactly one JSON line: NCCL's own banner / debug output goes to stderr
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        import torch
        import torch.distributed as dist_mod
        torch.cuda.set_device(local_rank)
        dist_mod.init_process_group("nccl")
        dist = dist_mod
    dev = local_rank
    comm = None
    if dist is not None:
        # one process per GPU: source rows sharded, NCCL exchange inside the library (unique id via torch)
        uid = [g.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        comm = (uid[0], rank, world)
    preprocessing = None
    if "raw" in wl:
        # raw scans -> device-resident pipeline (every rank pre-processes both scans on its own GPU: the stages are
        # deterministic, so all ranks hold identical keypoint sets; the registration below shards the source keypoints)
        Tc, Sc, _, _ = raw_scans(g, wl)
        best = None
        for _rep in range(2):                              # first pass = module load + allocator warm-up
            t0 = time.perf_counter()
            pt = g.Prep(Tc, wl["voxel"], wl["radius"], wl["nms"], bsc_radius=wl["nms"], dof_type=0, device=dev)
            ps = g.Prep(Sc, wl["voxel"], wl["radius"], wl["nms"], bsc_radius=wl["nms"], dof_type=wl["dof"], device=dev)
            wall_ms = (time.perf_counter() - t0) * 1e3
            if best is not None:
                best[0].close(); best[1].close()
            best = (pt, ps, wall_ms)
        pt, ps, wall_ms = best
        if ps.n_kp < 10 or pt.n_kp < 10:
            raise SystemExit("bench.py: the detector found too few keypoints")
        wl["N"], wl["M"] = ps.n_kp, pt.n_kp
        config.update(N_src=ps.n_kp, N_tgt=pt.n_kp, raw_points=[int(len(Sc)), int(len(Tc))])
        preprocessing = {"source": dict(points=int(len(Sc)), down=ps.n_down, keypoints=ps.n_kp, stage_ms=ps.stage_ms),
                         "target": dict(points=int(len(Tc)), down=pt.n_down, keypoints=pt.n_kp, stage_ms=pt.stage_ms),
                         "wall_ms_both_scans": wall_ms,
                         "raw_points_per_s": (len(Sc) + len(Tc)) / (ps.stage_ms["total"] + pt.stage_ms["total"]) * 1e3,
                         "note": "ghicp_prep_run: one upload per scan, voxel filter -> keypoints -> BSC chained on the device; "
                                 "stage_ms from CUDA events (h2d = the raw scan's host->device copy)"}
        t0 = time.perf_counter()
        Ef = g.Energyfunction().init(ps.n_kp, pt.n_kp, ps.bbx_magnitude)
        reg = g.GHRegistration((ps, pt), Ef, FT[wl["ft"]], CT[wl["ct"]], dof_type=wl["dof"], device=dev, comm=comm)
        t_upload = time.perf_counter() - t0
        S0 = np.asfortranarray(ps.keypoints()[1], dtype=np.float64)
        T_host = np.asfortranarray(pt.keypoints()[1], dtype=np.float64)
        pt.close(); ps.close()
    else:
        sc = make_scene(g, wl)
        t0 = time.perf_counter()
        reg = g.registration.from_scene(sc, FT[wl["ft"]], CT[wl["ct"]], device=dev, comm=comm)
        t_upload = time.perf_counter() - t0
        S0 = np.asfortranarray(sc.S, dtype=np.float64)
        T_host = np.asfortranarray(sc.T, dtype=np.float64)  # the reference holds kpTXYZ column-major (Eigen::MatrixX3d)
    t0 = time.perf_counter()
    reg.build_fd()
    t_fd = time.perf_counter() - t0

    def barrier():
        if dist is not None:
            dist.barrier()

    def allmax(x):
        if dist is None:
            return x
        import torch
        t = torch.tensor([x], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- a whole registration, iteration 0 .. convergence (device time per iteration, CUDA events inside the library):
    #      what a registration costs, dense first KM iterations included.  Run twice: the first pass also warms every
    #      allocation the dense iterations grow (edge buffers), the second is the one reported.
    REG_CAP = 60
    registration = None
    for _pass in range(2):
        reg.reset()
        reg.set_keypoints(S0, T_host)
        its = []
        for _ in range(REG_CAP):
            st = reg.iterate()
            its.append(dict(it=st.iteration, ms=st.ms_total, cor=st.cor, nnz=st.nnz, rounds=st.km_rounds, km_energy=st.km_energy))
            if st.converged:
                break
        total = allmax(float(sum(x["ms"] for x in its)))
        registration = dict(iterations=len(its), converged=bool(st.converged), ms_total=total, ms_per_iteration=total / len(its),
                            iterations_per_s=(1000.0 * len(its) / total) if total > 0 else None, first_iterations=its[:6],
                            note="device time of every iteration from 0 to convergence (max over ranks), second of two passes")

    # ---- warm-up: iterations 0..W-1 of a fresh registration; timed steps = iterations W..W+K-1 -----------------------
    reg.reset()
    reg.set_keypoints(S0, T_host)
    for _ in range(args.warmup):
        st = reg.iterate()

    # ---- timed region 1: device-resident steps -----------------------------------------------------
    launches = 0
    dev_ms, wall_ms, stage = [], [], []
    with ClockSampler(dev) as cs:
        time.sleep(0.05)   # the sampler thread's start-up (NVML handles) must not desynchronise the ranks' first timed step
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            t_step = time.perf_counter()
            st = reg.iterate()  # ends with a stream synchronize
            wall_ms.append((time.perf_counter() - t_step) * 1e3)
            dev_ms.append(st.ms_total)
            stage.append((st.ms_cost, st.ms_corr, st.ms_solve, st.nnz, st.km_rounds, st.cor, st.ms_stream,
                          st.stream_passes, st.exact_fallback, st.candidates))
            launches += st.gpu_launches
        wall = time.perf_counter() - t0
    barrier()
    clocks = cs.summary()
    ms_per_step = allmax(wall * 1e3 / args.steps)
    if args.dump_outputs and rank == 0:
        sp, tp = reg.pairs()
        dump_outputs(args.dump_outputs, {
            "source_pairs": sp, "target_pairs": tp, "source_keypoints": reg.source(), "rt_step": st.Rt_np(),
            "rt_accumulated": st.Rt_tillnow_np(),
            "stats": [st.iteration, st.cor, st.converged, st.penalty, st.rmse, st.rmse_after, st.fdm, st.fdstd, st.iou, st.para1,
                      st.para2, st.km_energy]})

    # ---- timed region 2: end to end through the host-facing API -----------------------------------
    # every step: host (pinned inside the library) -> device copy of the current source + target
    # coordinates, one iteration, device -> host read of the stats, the pair lists and the updated source.
    # host buffers of the end-to-end arm: page-locked (the bench contract's "pinned host memory"; ghicp_host_alloc), so every
    # copy below is one DMA straight from / into the caller's arrays
    S_host = g.capi.pinned_copy(reg.source(), order="F")
    T_pin = g.capi.pinned_copy(T_host, order="F")
    sp_buf = g.capi.pinned_empty(max(wl["N"], wl["M"]), np.int32)
    tp_buf = g.capi.pinned_empty(max(wl["N"], wl["M"]), np.int32)
    # time the same iteration range as the device-resident region (the weight schedule depends on the index)
    reg.set_state(args.warmup, st.rmse, st.fdm, st.fdstd, st.para1, st.para2)
    barrier()
    t0 = time.perf_counter()
    e2e_steps = args.steps
    for _ in range(e2e_steps):
        reg.set_keypoints(S_host, T_pin)
        st = reg.iterate()
        sp, tp = reg.pairs(out=(sp_buf, tp_buf))
        reg.source(out=S_host)
    e2e_wall = time.perf_counter() - t0
    barrier()
    e2e_ms = allmax(e2e_wall * 1e3 / e2e_steps)
    h2d = 24 * (wl["N"] + wl["M"])
    d2h = 24 * wl["N"] + 8 * int(st.cor) + 400

    if rank != 0:
        return
    hbm_peak, peak_src = peaks()
    # dominant kernel accounting (DESIGN.md §Roofline): the FD-plane stream of the cost stage
    stage = np.array(stage, dtype=np.float64)
    n_sweeps = int(np.median(stage[:, 7]))
    # algorithmic bytes of ONE streaming pass ON ONE GPU (SURVEY.md §8d): its rows of the fp16 FD plane once + the float4
    # operand arrays (16 B per keypoint) + 12 B per source row of results.  Sharded: rank 0 streams nloc = ceil(N/G) rows;
    # the kernel time is rank 0's, so both sides of achieved = bytes / time are per GPU.
    nloc = (wl["N"] + world - 1) // world
    alg_bytes = (2 * nloc * wl["M"] if wl["ft"] == "bsc" else 0) + 16 * (nloc + wl["M"]) + 12 * nloc
    cost_ms = float(np.median(stage[:, 0]))
    stream_ms = float(np.median(stage[:, 6]))
    achieved = alg_bytes / (stream_ms * 1e-3) / 1e9 if stream_ms > 0 else 0.0
    traffic = NCU_TRAFFIC.get(args.workload) if (not args.n and world == 1) else None
    roofline = {"kernel": "k_stream (calED+calCD+scan/gate+stats fused over the fp16 FD plane)", "bound": "hbm",
                "kernel_ms": stream_ms,
                "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak,
                "traffic": traffic["bytes"] if traffic else None, "traffic_source": traffic["source"] if traffic else None,
                "peak_source": peak_src, "per_gpu": True, "rows_per_gpu": nloc,
                "algorithmic_bytes_per_launch": alg_bytes, "sweeps_per_step": n_sweeps}
    if wl["ft"] == "fpfh":
        # matrix-free FPFH: O(N+M) bytes for N*M pair evaluations -> the FP32 pipe, not HBM, bounds the sweep.
        # Dominant kernel = k_ff_sweep<MAIN> (FP32 filter; ms_stream is its CUDA-event time).  Algorithmic work per pair
        # (DESIGN.md §3.5): 33 FFMA (histogram dot) + 12 (hi/lo coordinate differences, d2) + 8 (cost, bound, sum) = 53
        # FP32-pipe instructions; peak = 148 SMs x 128 lanes x SM clock.
        pairs = float(nloc) * wl["M"]
        fast = stream_ms > 0
        t_ms = stream_ms if fast else cost_ms
        sm_mhz = (clocks.get("sm_mhz") or 1965.0)
        peak_ginstr = 148 * 128 * sm_mhz * 1e6 / 1e9
        ach = 53.0 * pairs / (t_ms * 1e-3) / 1e9 if t_ms > 0 else 0.0
        roofline = {"kernel": "k_ff_sweep (FP32 filter over on-the-fly FPFH distances + exact FP64 refinement)" if fast
                    else "k_rowsweep_mf / k_colsweep_mf (exact all-double matrix-free sweeps)",
                    "bound": "fp32-pipe", "kernel_ms": t_ms, "achieved": ach if fast else None, "peak": peak_ginstr,
                    "unit": "Ginstr/s", "frac": (ach / peak_ginstr) if fast else None, "traffic": None,
                    "pairs_per_s": pairs / (t_ms * 1e-3) if t_ms > 0 else 0.0, "sweeps_per_step": n_sweeps,
                    "algorithmic_instr_per_pair": 53, "per_gpu": True}
    line = {
        "metric": "ICP iterations/sec", "value": 1000.0 / ms_per_step,
        "unit": "iterations/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic", "config": config,
        "value_is": f"iterations {args.warmup}..{args.warmup + args.steps - 1} of a registration (settled regime); "
                    "`registration` holds the whole-registration figure, dense first iterations included",
        "registration": registration,
        "device_ms_per_step": float(np.mean(dev_ms)),
        # rank 0's view of every timed step: CUDA-event time of the iteration, wall time of the ghicp_iterate call
        "per_step": {"device_ms": [round(x, 3) for x in dev_ms], "wall_ms": [round(x, 3) for x in wall_ms]},
        "stage_ms": {"cost": cost_ms, "corr": float(np.median(stage[:, 1])), "solve": float(np.median(stage[:, 2]))},
        "km": {"nnz": int(np.median(stage[:, 3])), "rounds": int(np.median(stage[:, 4]))} if km else None,
        "cor": int(stage[-1, 5]),
        "first_iterations": registration["first_iterations"],
        "one_time": {"fd_build_s": t_fd, "upload_s": t_upload},
        "preprocessing": preprocessing,
        "e2e": {"value": 1000.0 / e2e_ms, "unit": "iterations/s", "ms_per_step": e2e_ms,
                "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
        "gpu_launches": launches,
        "clocks": clocks,
        "exact_fallbacks": int(stage[:, 8].sum()), "filter_candidates_per_step": int(np.median(stage[:, 9])),
        "roofline": roofline,
    }
    if not args.no_cpu:
        # bounded CPU sample, the same iteration indices as the timed region (10-30 s of CPU work)
        if "raw" in wl:
            cap = args.cpu_sample or 125000
            sizes = [min(wl["raw"], cap // 2), min(wl["raw"], cap)]
        elif wl["N"] <= 1500:
            sizes = [wl["N"]]
        else:
            n_s = args.cpu_sample or (1500 if km else 4000)
            sizes = [max(400, n_s // 2), min(n_s, wl["N"])]
        cb = cpu_arm(g, wl, args.warmup, min(args.steps, 4), sizes, fit_steps=2)
        line["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample", "extrapolated", "fit", "registration")}
        try:   # SURVEY.md §8d "fair CPU": the O(N*M) loops on all host cores (OpenMP), KM serial (it is sequential as written)
            th = min(ncores, 8)
            fc = cpu_arm(g, wl, args.warmup, min(args.steps, 4), [sizes[-1]], threads=th)
            line["cpu_baseline"]["fair_cpu"] = {"cores": th, "kind": fc["kind"], "sample_n": fc["sample_n"],
                                                "ms_per_iteration_sample": fc["ms_per_step_sample"],
                                                "single_thread_ms_per_iteration_sample": cb["ms_per_step_sample"]}
        except Exception as e:  # the OpenMP oracle is optional test infrastructure
            line["cpu_baseline"]["fair_cpu"] = {"unavailable": str(e)[:200]}
    emit(line)


if __name__ == "__main__":
    main()
