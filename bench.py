#!/usr/bin/env python
"""bench.py — filter-steps/s of the batched 1-point-RANSAC EKF-SLAM filter step on B200.

Contract: ``python bench.py --gpus N --steps K --warmup W`` (under torchrun for N>1) prints ONE
JSON line from rank 0.  A "step" is one pass of the whole filter step (mc/mono_slam.m:56-74:
predict -> h/H/S -> matcher gate -> 1-point RANSAC -> li update -> rescue -> hi update) over a
batch of independent Monte-Carlo filters; workload = BASELINE.json configs[2]: N=100 inverse-depth
features, 4096 filters per GPU (weak scaling: every rank owns its own 4096 filters, no data-path
collective; NCCL only gathers per-filter statistics after the timed region).

  value  = filter-steps/s with the frame inputs already resident in HBM (kernel path only)
  e2e    = the same through the host-buffer C-ABI call (ekfslam_step_host): per step the frame's
           candidate pixels + flags + RANSAC uniforms go host->device from pinned memory and the
           new camera/feature state x_k_k, the inlier flags and the step statistics come back.
  roofline / cpu_baseline: see DESIGN.md §Measurement.

``--impl reference`` times the CPU oracle port of the reference (the reference itself is MATLAB
and cannot run here: no Octave/MATLAB in the image) on the host cores, on the same workload.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "filter-steps/s at N=100 features, batch 4096 filters"
UNIT = "filter-steps/s"


def workload_name(features, batch):
    """config.workload, identical in the repo arm and the reference arm (BASELINE.json configs[2])."""
    return ("cfg3: N=%d inverse-depth features (n=%d), batch %d Monte-Carlo filters per GPU, synthetic point-field "
            "sequence" % (features, 13 + 6 * features, batch))


def cpu_sample_filters(threads, override=0):
    """Filters per step of the bounded CPU sample (same definition in `cpu_baseline` and `--impl reference`)."""
    return override or min(16 * threads, 512)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=4)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=4096, help="filters per GPU")
    ap.add_argument("--features", type=int, default=100)
    ap.add_argument("--fixed-hyp", type=int, default=0, help="0 = reference adaptive rule; >0 = fixed budget")
    ap.add_argument("--n-u", type=int, default=0, help="uniforms per frame (default 64 adaptive / fixed-hyp)")
    ap.add_argument("--p-outlier", type=float, default=0.2)
    ap.add_argument("--seed", type=int, default=2024)
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-sample", type=int, default=0, help="filters in the CPU sample (0 = auto)")
    ap.add_argument("--no-extra", action="store_true", help="skip the cfg4 / strong-split / sustained extras")
    ap.add_argument("--sustained-steps", type=int, default=60)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the state the last timed device-resident step left (x_k_k, inlier flags, step "
                         "statistics, a sample of P_k_k) of rank 0 to DIR/<name>.npy; see dump_outputs()")
    return ap.parse_args()


# ------------------------------------------------------------------------------------------
# algorithmic work (SURVEY.md §8d / BASELINE.md §4), per filter
# ------------------------------------------------------------------------------------------
def algorithmic_work(n, N, m, hyps, k_li, k_hi):
    upd_b = sum(2 * n * n + 2 * n * k for k in (k_li, k_hi))
    nbytes = 8.0 * (52 * n + 2 * (n + 201 * N) + n * n + upd_b)
    upd_f = sum(n * n * k + n * k * k + k ** 3 / 3.0 + 26 * n * k + 26 * k * k for k in (k_li, k_hi))
    flops = 676.0 * n + 3504.0 * N + hyps * (56.0 * n + 200.0 * m) + upd_f
    return nbytes, flops


def read_traffic(kernel_prefix):
    """dram__bytes_read+write per launch of a kernel from the committed ncu capture of this shape."""
    p = os.path.join(ROOT, "profiles", "ncu_traffic_r2h.json")
    try:
        with open(p) as f:
            d = json.load(f)
        rows = [x for k, v in d["kernels"].items() if k.startswith(kernel_prefix) for x in v]
        if rows:
            return sum(x["dram_read"] + x["dram_write"] for x in rows) / len(rows)
    except Exception:
        pass
    return None


def read_peaks():
    peaks = {"hbm_gbs": 6650.0, "hbm_src": "fallback (B200_PROFILING.md)", "fp64_tflops": 37.0,
             "fp64_src": "nominal (no measurement found)"}
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            with open(p) as f:
                peaks["hbm_gbs"] = float(json.load(f)["hbm_gbs"])
            peaks["hbm_src"] = "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    p = os.path.join(ROOT, "profiles", "fp64_peak.json")
    if os.path.exists(p):
        try:
            with open(p) as f:
                d = json.load(f)
            peaks["fp64_tflops"] = float(max(d["dfma_tflops"], d["dmma_m8n8k4_tflops"]))
            peaks["fp64_src"] = "measured (profiles/fp64_peak.json, tools/microbench_fp64.cu)"
        except Exception:
            pass
    return peaks


class ClockSampler:
    """SM clock, power and throttle reasons sampled every 50 ms for the duration of the timed regions.  NVML is
    queried in-process from a thread (nvidia_ml_py): a polling `nvidia-smi -lms` process stalls the driver for
    milliseconds per sample, which the synchronous host-buffer (e2e) steps pay in full (measured: +5 ms per step).
    Falls back to one long-lived `nvidia-smi -lms 250` when NVML cannot be loaded."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.samples = []
        self.thread = None
        self.stop_flag = False

    def _nvml_loop(self, nv, h):
        smax = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
        R = nv
        while not self.stop_flag:
            try:
                sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
                pw = nv.nvmlDeviceGetPowerUsage(h) / 1000.0
                rs = nv.nvmlDeviceGetCurrentClocksEventReasons(h) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                    else nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                flag = lambda bit: "Active" if (rs & bit) else "Not Active"  # noqa: E731
                self.samples.append([str(sm), str(smax), "%.2f" % pw,
                                     flag(getattr(R, "nvmlClocksThrottleReasonHwSlowdown", 0x8)),
                                     flag(getattr(R, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40)),
                                     flag(getattr(R, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20)),
                                     flag(getattr(R, "nvmlClocksThrottleReasonSwPowerCap", 0x4))])
            except Exception:
                pass
            time.sleep(0.05)

    def start(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            # NVML enumerates all GPUs of the box; CUDA_VISIBLE_DEVICES may remap the CUDA ordinal
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = self.index
            if vis:
                ids = [v.strip() for v in vis.split(",") if v.strip()]
                if self.index < len(ids) and ids[self.index].isdigit():
                    idx = int(ids[self.index])
            h = nv.nvmlDeviceGetHandleByIndex(idx)
            import threading
            self.thread = threading.Thread(target=self._nvml_loop, args=(nv, h), daemon=True)
            self.thread.start()
            return
        except Exception:
            self.thread = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "250"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        if self.thread is not None:
            self.stop_flag = True
            self.thread.join(timeout=2)
            return
        if self.proc is None:
            return
        try:
            self.proc.terminate()
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            out = ""
        for line in out.splitlines():
            parts = [p.strip() for p in line.split(",")]
            if len(parts) >= 7 and parts[0].replace(".", "", 1).isdigit():
                self.samples.append(parts)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm = sorted(float(s[0]) for s in self.samples)
        reasons = []
        for i, name in enumerate(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]):
            if any(s[3 + i].lower().startswith("active") for s in self.samples):
                reasons.append(name)
        pw = [float(s[2]) for s in self.samples if s[2].replace(".", "", 1).isdigit()]
        return {"sm_mhz": sm[len(sm) // 2], "sm_min_mhz": sm[0], "sm_max_mhz": float(self.samples[0][1]),
                "reasons": reasons, "samples": len(sm), "power_w_max": max(pw) if pw else None}


# ------------------------------------------------------------------------------------------
# CPU arm: the oracle port on host cores (oracle/ekf_oracle.c, OpenMP over filters)
# ------------------------------------------------------------------------------------------
def host_cores():
    return len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)


def cpu_reference_rate(args, n_filters, steps, warm, threads):
    """filter-steps/s of the C oracle: `n_filters` filters x `steps` timed steps on `threads` threads."""
    import ekf_slam_b200.synth as synth
    from oracle import c_oracle
    n_u = args.n_u or (args.fixed_hyp if args.fixed_hyp > 0 else 64)
    seq = synth.SynthSequence(B=n_filters, N=args.features, T=warm + steps, seed=args.seed,
                              p_outlier=args.p_outlier, n_u=n_u)
    x, P, types = seq.initial_state()
    nfeat = np.full(n_filters, args.features, dtype=np.int32)
    wall = 0.0
    for t in range(1, warm + steps + 1):
        zc = np.ascontiguousarray(seq.zc[t])
        has = np.ascontiguousarray(seq.has[t])
        u = seq.uniforms(t, n_u)
        t0 = time.perf_counter()
        c_oracle.step_batch(x, P, types, nfeat, zc, has, u, fixed_hyp=args.fixed_hyp, nthreads=threads)
        if t > warm:
            wall += time.perf_counter() - t0
    return n_filters * steps / wall, wall


def octave_probe():
    """SURVEY §8(d): the number north_star asks for is the reference under GNU Octave.  Probe for it; when absent say so
    (never a made-up number).  When present, baseline/octave/run_ref_step.m runs the unmodified reference functions."""
    import shutil
    exe = shutil.which("octave")
    if exe is None:
        sys.stderr.write("OCTAVE ABSENT - reference CPU path (GNU Octave) not measured; timing the C port instead\n")
        return {"octave": None, "note": "OCTAVE ABSENT - reference CPU path not measured"}
    ref = "/root/reference/matlab_code"
    here = os.path.join(os.path.dirname(os.path.abspath(__file__)), "baseline", "octave")
    if not os.path.isdir(ref):
        return {"octave": exe, "note": "octave present but the reference sources are not on this box"}
    import subprocess, tempfile, importlib.util
    spec = importlib.util.spec_from_file_location("export_inputs", os.path.join(here, "export_inputs.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    with tempfile.TemporaryDirectory() as td:
        inp, outp = os.path.join(td, "in.mat"), os.path.join(td, "out.mat")
        mod.export(inp, 2, 100, 3)
        r = subprocess.run([exe, "--no-gui", "--quiet", "--eval",
                            "addpath('%s'); run_ref_step('%s','%s','%s')" % (here, inp, outp, ref)],
                           capture_output=True, text=True, timeout=1200)
        rate = None
        for ln in r.stdout.splitlines():
            if ln.startswith("REFERENCE"):
                rate = float(ln.split("=")[1].split()[0])
        return {"octave": exe, "filter_steps_per_s": rate, "sample": "2 filters x 3 steps, N=100, single Octave process"}


def run_reference(args, rank):
    """The CPU arm: the reference's algorithm on the host cores.  GNU Octave / MATLAB are absent in this image, so the
    arm times the C restatement of the reference (oracle/ekf_oracle.c; pinned against the reference's own execution,
    tests/test_oracle_ref.py) with all host threads.  Each step processes a BOUNDED SAMPLE of the batch
    (`cpu_baseline.sample`); `ms_per_step` is the measured time of such a step, `value` the throughput."""
    if rank != 0:
        return
    octave = octave_probe()
    threads = max(1, min(host_cores(), 256))
    nf = cpu_sample_filters(threads, args.cpu_sample)
    steps, warm = max(1, args.steps), max(1, min(args.warmup, 3))
    rate, wall = cpu_reference_rate(args, nf, steps, warm, threads)
    sample = ("%d filters per step x %d timed steps (+%d warm-up) of the same synthetic workload, C restatement "
              "oracle/ekf_oracle.c, OpenMP %d threads, %.1f s timed" % (nf, steps, warm, threads, wall))
    line = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * wall / steps,
        "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": {"workload": workload_name(args.features, args.batch),
                   "filters_per_step_in_this_arm": nf,
                   "ms_per_step_note": "measured time of one step over the bounded sample of %d filters (not the "
                                       "full batch of %d)" % (nf, args.batch),
                   "ransac": "adaptive (reference rule)" if args.fixed_hyp <= 0 else "fixed %d" % args.fixed_hyp,
                   "p_outlier": args.p_outlier,
                   "reference_runtime": "GNU Octave / MATLAB absent in this image: C port of the reference "
                                        "(oracle/ekf_oracle.c) on all host cores"},
        "cpu_baseline": {"value": rate, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "octave": octave,
    }
    emit(line)



# ------------------------------------------------------------------------------------------
# extras: other BASELINE configs under the driver's eyes (same process, same box, a few steps each)
# ------------------------------------------------------------------------------------------
def run_resident(pkg, synth, torch, dev, device_index, B, N, warm, timed, seed, b_offset=0, fixed_hyp=0, barrier=None):
    """B filters of N features: map built on the device, frames resident in HBM, `warm` untimed + `timed` timed
    steps on a private stream.  Returns (ms_total, kernel_times, stats, mean state size)."""
    n_u = fixed_hyp if fixed_hyp > 0 else 64
    T = warm + timed
    seq = synth.SynthSequence(B=B, N=N, T=T, seed=seed, b_offset=b_offset, n_u=n_u)
    bank = pkg.FilterBank(B, N, device=device_index)
    stream = torch.cuda.Stream(dev)
    bank.set_stream(stream.cuda_stream)
    bank.set_params(fixed_hyp=fixed_hyp)
    bank.reset_filters()
    for k in range(N):
        bank.add_features_inverse_depth(np.ascontiguousarray(seq.zc[0, :, k]))
    zc = torch.from_numpy(seq.zc).to(dev)
    fl = torch.from_numpy((seq.has * pkg.F_CAND).astype(np.uint8)).to(dev)
    u = torch.from_numpy(np.ascontiguousarray(np.transpose(seq.U, (1, 0, 2)))).to(dev)
    torch.cuda.synchronize(dev)

    def step(t):
        bank.bind_frame(zc[t].data_ptr(), fl[t].data_ptr(), u[t].data_ptr(), n_u)
        bank.step(reset=True, match_mode=1)

    for t in range(1, warm + 1):
        step(t)
    torch.cuda.synchronize(dev)
    bank.enable_timing(True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if barrier:
        barrier()
    torch.cuda.synchronize(dev)
    e0.record(stream)
    for t in range(warm + 1, T + 1):
        step(t)
    e1.record(stream)
    torch.cuda.synchronize(dev)
    if barrier:
        barrier()
    ms = e0.elapsed_time(e1)
    kt = {k: v[0] / timed for k, v in bank.kernel_times().items() if v[1] > 0}
    st = bank.download_stats()
    _, _, ns = bank.download_state(want_P=False)
    bank.unbind_frame()
    bank.close()
    del zc, fl, u
    return ms, kt, st, float(ns.mean())


def extra_cfg4(pkg, synth, torch, dev, device_index, peaks):
    """BASELINE configs[3]: large map N=500 (n=3013), batch 8 - the dense covariance downdate on the fp64 tensor pipe."""
    B, N, warm, timed = 8, 500, 2, 4
    ms, kt, st, n = run_resident(pkg, synth, torch, dev, device_index, B, N, warm, timed, seed=1)
    k_li, k_hi = 2.0 * float(st["n_li"].mean()), 2.0 * float(st["n_hi"].mean())
    out = {"workload": "cfg4: large map N=500 (n=%d), batch %d, adaptive RANSAC" % (int(n), B), "B": B, "N": N,
           "steps": timed, "warmup": warm, "ms_per_step": ms / timed, "filter_steps_per_s": B * timed / (ms * 1e-3),
           "mean_k_li": k_li, "mean_k_hi": k_hi, "chol_ms": kt.get("k_chol", 0.0), "chol_hi_ms": kt.get("k_chol_hi", 0.0),
           "kernels_ms_per_step": {k: round(v, 4) for k, v in sorted(kt.items(), key=lambda kv: -kv[1])},
           "status_flags": int((st["status"] != 0).sum())}
    if kt.get("k_downdate"):
        tf = B * n * n * k_li / (kt["k_downdate"] * 1e-3) / 1e12     # n^2 k flops of the lower-triangle downdate (FMA = 2)
        out.update({"li_downdate_ms": kt["k_downdate"], "li_downdate_tflops": tf,
                    "frac_of_dmma_peak": tf / peaks["fp64_tflops"], "dmma_peak_tflops": peaks["fp64_tflops"],
                    "dmma_peak_source": peaks["fp64_src"]})
    return out


DUMP_BYTES = 60_000_000   # stays under 64 MB in all, with room for the index arrays


def dump_outputs(bank, out_dir):
    """Writes what a caller of the step receives after the last timed step, so that two builds can be compared output
    for output on the same seeded workload:
      x.npy [F, n_max] f64 (x_k_k), flags.npy [F, N] f32 (inlier flag bits), stats.npy [F, 8] f64 (the per-filter step
      statistics, columns in the order of include/ekfslam.h) for the filters in filters.npy;
      P.npy [G, R, n_max] f64 (rows P_rows.npy of P_k_k) for the filters in P_filters.npy.
    Every filter and every row is kept when it fits half of DUMP_BYTES each; otherwise a fixed, seeded sample."""
    from ekf_slam_b200._lib import STATS_FIELDS
    os.makedirs(out_dir, exist_ok=True)
    rng = np.random.default_rng(0)
    B, N, n = bank.B, bank.N, bank.n_max
    half = DUMP_BYTES // 2

    def sample(total, keep):
        return np.arange(total) if keep >= total else np.sort(rng.choice(total, keep, replace=False))

    filters = sample(B, half // (8 * n + 4 * N + 8 * len(STATS_FIELDS)))
    x, _, _ = bank.download_state(want_P=False)
    st = bank.download_stats()
    out = {"filters": filters, "x": x[filters], "flags": bank.download_flags()[filters].astype(np.float32),
           "stats": np.stack([st[k] for k in STATS_FIELDS], axis=1)[filters]}
    p_filters = sample(B, max(1, half // (8 * n * n)))
    rows = sample(n, half // (8 * n * len(p_filters)))
    out.update(P_filters=p_filters, P_rows=rows,
               P=np.stack([bank.download_state(b0=int(b), nb=1)[1][0][rows] for b in p_filters]))
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a if a.dtype in (np.float32, np.float64) else a.astype(np.float64))


# ------------------------------------------------------------------------------------------
_REAL_STDOUT = None


def emit(line):
    """Exactly one JSON line on the real stdout (everything else — NCCL banners, torchrun notices —
    was redirected to stderr at start-up)."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    global _REAL_STDOUT
    args = parse()
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)  # library chatter on fd 1 (e.g. "NCCL version ...") goes to stderr
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return

    import torch
    import torch.distributed as dist
    import ekf_slam_b200 as pkg
    import ekf_slam_b200.synth as synth

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    if world != args.gpus and rank == 0:
        print("warning: --gpus %d but WORLD_SIZE %d" % (args.gpus, world), file=sys.stderr)

    K, W, N = args.steps, args.warmup, args.features
    B = args.batch if args.scaling == "weak" else max(1, args.batch // world)
    n = 13 + 6 * N
    n_u = args.n_u or (args.fixed_hyp if args.fixed_hyp > 0 else 64)
    We = min(W, 3) if not args.no_e2e else 0   # untimed warm-up steps of the host-buffer path (its own streams / copies)
    Ks = 0 if args.no_extra else max(0, args.sustained_steps)   # extra: a longer device-resident window
    T = W + 2 * K + We + Ks
    t_setup = time.perf_counter()
    seq = synth.SynthSequence(B=B, N=N, T=T, seed=args.seed, b_offset=rank * B, p_outlier=args.p_outlier, n_u=n_u)
    bank = pkg.FilterBank(B, N, n, device=local_rank)
    # a dedicated non-default stream shared by torch (events) and the library (kernels, copies)
    stream = torch.cuda.Stream(dev)
    torch.cuda.set_stream(stream)
    assert stream.cuda_stream != 0
    bank.set_stream(stream.cuda_stream)
    bank.set_params(fixed_hyp=args.fixed_hyp)
    # frame-0 map built ON THE DEVICE from the first observations (mc/initialize_x_and_p.m, then
    # mc/add_features_inverse_depth.m once per feature) — no 12 GB host covariance to upload
    bank.reset_filters()
    for k in range(N):
        bank.add_features_inverse_depth(np.ascontiguousarray(seq.zc[0, :, k]))
    # frame inputs: pinned host copies (e2e arm) and HBM-resident copies (device arm)
    fl_np = (seq.has * pkg.F_CAND).astype(np.uint8)
    zc_pin = torch.from_numpy(seq.zc).pin_memory()
    fl_pin = torch.from_numpy(fl_np).pin_memory()
    u_pin = torch.from_numpy(np.ascontiguousarray(np.transpose(seq.U, (1, 0, 2)))).pin_memory()   # [T+1,B,n_u]
    zc_dev = zc_pin.to(dev)
    fl_dev = fl_pin.to(dev)
    u_dev = u_pin.to(dev)
    torch.cuda.synchronize(dev)
    t_setup = time.perf_counter() - t_setup

    def bind(t):
        bank.bind_frame(zc_dev[t].data_ptr(), fl_dev[t].data_ptr(), u_dev[t].data_ptr(), n_u)

    def barrier():
        if world > 1:
            dist.barrier()

    # ---- warm-up (also lets the covariances fill in) -------------------------------------
    for t in range(1, W + 1):
        bind(t)
        bank.step(reset=True, match_mode=1)
    torch.cuda.synchronize(dev)

    # ---- timed region: device-resident inputs ----------------------------------------------
    sampler = ClockSampler(local_rank)
    sampler.start()
    bank.enable_timing(True)
    l0 = bank.launch_count
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    torch.cuda.synchronize(dev)
    ev0.record(stream)
    for t in range(W + 1, W + K + 1):
        bind(t)
        bank.step(reset=True, match_mode=1)
    ev1.record(stream)
    torch.cuda.synchronize(dev)
    barrier()
    ms_dev = ev0.elapsed_time(ev1)
    launches = bank.launch_count - l0
    ktimes = bank.kernel_times()
    bank.enable_timing(False)
    stats = bank.download_stats()
    bank.unbind_frame()
    if args.dump_outputs and rank == 0:
        dump_outputs(bank, args.dump_outputs)

    # ---- timed region: end to end through the host-buffer call ------------------------------
    e2e = None
    if not args.no_e2e:
        x_out = torch.empty((B, n), dtype=torch.float64).pin_memory()
        f_out = torch.empty((B, N), dtype=torch.uint8).pin_memory()
        s_out = torch.empty((B, 8), dtype=torch.int32).pin_memory()
        zc_h, fl_h, u_h = zc_pin.numpy(), fl_pin.numpy(), u_pin.numpy()
        xo, fo, so = x_out.numpy(), f_out.numpy(), s_out.numpy()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for t in range(W + K + 1, W + K + We + 1):   # warm-up of the host-buffer call (first-use costs of its copy path)
            bank.step_host(zc_h[t], fl_h[t], u_h[t], match_mode=1, x_out=xo, flags_out=fo, stats_out=so)
        barrier()
        torch.cuda.synchronize(dev)
        e0.record(stream)
        for t in range(W + K + We + 1, W + 2 * K + We + 1):
            bank.step_host(zc_h[t], fl_h[t], u_h[t], match_mode=1, x_out=xo, flags_out=fo, stats_out=so)
        e1.record(stream)
        torch.cuda.synchronize(dev)
        barrier()
        ms_e2e = e0.elapsed_time(e1)
        h2d = zc_h[1].nbytes + fl_h[1].nbytes + u_h[1].nbytes
        d2h = xo.nbytes + fo.nbytes + so.nbytes
        e2e = (ms_e2e, h2d, d2h)
    # ---- extras (not the headline): sustained window, strong split of the 4096-filter batch ----------------
    extra = {}
    if Ks > 0:
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        torch.cuda.synchronize(dev)
        s0.record(stream)
        for t in range(T - Ks + 1, T + 1):
            bind(t)
            bank.step(reset=True, match_mode=1)
        s1.record(stream)
        torch.cuda.synchronize(dev)
        barrier()
        bank.unbind_frame()
        ms_sus = s0.elapsed_time(s1)
    sampler.stop()
    import ekf_slam_b200.sharding as sharding
    if Ks > 0:
        ms_sus = sharding.max_over_ranks(ms_sus, device=dev)
        extra["sustained"] = {"steps": Ks, "ms_per_step": ms_sus / Ks, "value": B * world * Ks / (ms_sus * 1e-3),
                              "window_s": ms_sus * 1e-3,
                              "note": "frames %d..%d of the same sequences, device-resident inputs; later frames carry "
                                      "fewer high-innovation inliers, so steps get cheaper" % (T - Ks + 1, T)}
    if not args.no_extra:
        # BASELINE configs[2] as written: 4096 filters TOTAL sharded over the ranks (strong scaling)
        if world == 1 or args.scaling == "strong":
            extra["strong"] = {"filters_total": args.batch if args.scaling == "weak" else B * world, "filters_per_gpu": B,
                               "note": "identical to the headline run at this N / scaling"}
        else:
            Bs = max(1, args.batch // world)
            ms_s, _, _, _ = run_resident(pkg, synth, torch, dev, local_rank, Bs, N, 3, K, seed=args.seed,
                                         b_offset=rank * Bs, fixed_hyp=args.fixed_hyp, barrier=barrier)
            ms_s = sharding.max_over_ranks(ms_s, device=dev)
            extra["strong"] = {"filters_total": Bs * world, "filters_per_gpu": Bs, "steps": K, "ms_per_step": ms_s / K,
                               "value": Bs * world * K / (ms_s * 1e-3)}

    # ---- reduce over ranks (max time), gather per-filter statistics over NCCL ---------------
    ms_dev = sharding.max_over_ranks(ms_dev, device=dev)
    ms_e2e = sharding.max_over_ranks(e2e[0] if e2e else 0.0, device=dev)
    tot_filters = B * world
    allst = sharding.gather_stats(stats, n_filters_total=tot_filters, device=dev)
    svec = [float(allst["n_li"].sum()), float(allst["n_hi"].sum()), float(allst["n_ic"].sum()),
            float(allst["ransac_iters"].sum()), float(allst["ransac_scored"].sum()),
            float((allst["status"] != 0).sum())]
    mean = lambda i: svec[i] / tot_filters  # noqa: E731

    if rank == 0:
        peaks = read_peaks()
        value = tot_filters * K / (ms_dev * 1e-3)
        k_li, k_hi = 2 * mean(0), 2 * mean(1)
        m, hyps = mean(2), mean(3)
        nbytes, flops = algorithmic_work(n, N, m, hyps, k_li, k_hi)
        # dominant kernel = the covariance downdate P -= W'W (two launches per step: li and hi)
        kt = {k: v for k, v in ktimes.items() if v[1] > 0}
        tot_k_ms = sum(v[0] for v in kt.values())
        top = max(kt.items(), key=lambda kv: kv[1][0])
        dd_li, dd_hi = kt.get("k_downdate", (0.0, 0)), kt.get("k_downdate_hi", (0.0, 0))
        dd_ms, dd_cnt = dd_li[0] + dd_hi[0], dd_li[1] + dd_hi[1]
        # per launch (whole batch B): flops n^2 k (lower triangle, FMA = 2) over the rows it applies, bytes 2 n^2 * 8;
        # two launches per step (li and hi update)
        dd_launches_per_step = dd_cnt / float(K) if dd_cnt else float("nan")
        dd_flops_per_step = B * sum(n * n * k for k in (k_li, k_hi))
        dd_bytes_per_step = B * dd_launches_per_step * (2 * n * n * 8.0)
        dd_s_per_step = (dd_ms * 1e-3) / K if dd_cnt else float("nan")
        dd_tf = dd_flops_per_step / dd_s_per_step / 1e12
        dd_gbs = dd_bytes_per_step / dd_s_per_step / 1e9
        t_fp = dd_flops_per_step / (peaks["fp64_tflops"] * 1e12)
        t_hbm = dd_bytes_per_step / (peaks["hbm_gbs"] * 1e9)
        if t_fp >= t_hbm:
            roof = {"bound": "tensor", "achieved": dd_tf, "peak": peaks["fp64_tflops"], "unit": "TFLOP/s",
                    "frac": dd_tf / peaks["fp64_tflops"], "traffic": None,
                    "peak_source": "fp64 " + peaks["fp64_src"]}
        else:
            roof = {"bound": "hbm", "achieved": dd_gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                    "frac": dd_gbs / peaks["hbm_gbs"], "traffic": None, "peak_source": "hbm " + peaks["hbm_src"]}
        if B == 4096 and N == 100:
            roof["traffic"] = read_traffic("k_downdate")
            roof["traffic_source"] = ("profiles/ncu_traffic_r2h.json (committed ncu --set full capture of this command at this shape, frame 3; "
                                      "mean of the li and hi launches) - not re-measured in this run")
        roof.update({"kernel": "k_downdate", "kernel_share_of_step": dd_ms / tot_k_ms if tot_k_ms else None,
                     "kernel_ms_per_launch": dd_ms / dd_cnt if dd_cnt else None, "launches_timed": dd_cnt,
                     "launches_per_step": dd_launches_per_step,
                     "algorithmic_flops_per_launch": dd_flops_per_step / dd_launches_per_step,
                     "algorithmic_bytes_per_launch": dd_bytes_per_step / dd_launches_per_step,
                     "hbm_gbs_achieved": dd_gbs, "fp64_tflops_achieved": dd_tf})
        step_roof = {"bytes_per_filter_step": nbytes, "flops_per_filter_step": flops,
                     "hbm_frac_of_step": (nbytes * tot_filters * K / world / (ms_dev * 1e-3)) / (peaks["hbm_gbs"] * 1e9),
                     "fp64_frac_of_step": (flops * tot_filters * K / world / (ms_dev * 1e-3)) / (peaks["fp64_tflops"] * 1e12)}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms_dev / K, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_name(N, args.batch), "p_outlier": args.p_outlier,
                       "filters_per_gpu": B, "global_batch": tot_filters,
                       "ransac": "adaptive (reference rule)" if args.fixed_hyp <= 0 else "fixed %d" % args.fixed_hyp,
                       "parallelism": "filters sharded across ranks, no data-path collective",
                       "l2": "inputs larger than L2 (covariances %.1f GB per GPU vs 126 MB L2)" % (B * n * n * 8 / 1e9),
                       "mean_matches": m, "mean_li_inliers": mean(0), "mean_hi_inliers": mean(1),
                       "mean_hypotheses_drawn": hyps, "mean_hypotheses_scored": mean(4),
                       "filters_with_status_flags": int(svec[5]), "setup_s": t_setup},
            "gpu_launches": int(launches),
            "roofline": roof,
            "step_roofline": step_roof,
            "kernels_ms_per_step": {k: v[0] / K for k, v in sorted(kt.items(), key=lambda kv: -kv[1][0])},
            "top_kernel": top[0],
            "ransac_hyps_per_s": {"drawn": hyps * tot_filters * K / (ms_dev * 1e-3),
                                  "scored": mean(4) * tot_filters * K / (ms_dev * 1e-3),
                                  "kernel_only_drawn": (hyps * B * K / (kt["k_ransac"][0] * 1e-3)) if "k_ransac" in kt else None},
            "clocks": sampler.summary(),
        }
        if e2e:
            line["e2e"] = {"value": tot_filters * K / (ms_e2e * 1e-3), "unit": UNIT,
                           "h2d_bytes_per_step": int(e2e[1]), "d2h_bytes_per_step": int(e2e[2]),
                           "ms_per_step": ms_e2e / K,
                           "note": "covariances stay resident on the device between frames (filter state, like the "
                                   "reference's persistent `filter` struct); per-frame inputs/outputs cross PCIe"}
        if "strong" in extra:
            st_ = extra["strong"]
            if "value" not in st_:
                st_.update({"value": value, "ms_per_step": ms_dev / K})
            # ideal strong value at N ranks = N x the single-GPU rate = this run's weak value (weak efficiency ~ 1)
            st_["efficiency_vs_weak_value"] = st_["value"] / value
        if not args.no_extra:
            try:
                extra["cfg4"] = extra_cfg4(pkg, synth, torch, dev, local_rank, peaks)
            except Exception as e:  # the extras never take the headline down
                extra["cfg4"] = {"error": repr(e)}
        if extra:
            line["extra"] = extra
        if not args.no_cpu_baseline:
            threads = max(1, min(host_cores(), 256))
            nf = cpu_sample_filters(threads, args.cpu_sample)
            rate, wall = cpu_reference_rate(args, nf, 6, 1, threads)
            line["cpu_baseline"] = {"value": rate, "unit": UNIT, "cores": threads, "kind": "port",
                                    "sample": "%d filters per step x 6 timed steps (+1 warm-up) of the same synthetic "
                                              "workload, C restatement oracle/ekf_oracle.c, OpenMP %d threads, %.1f s "
                                              "timed" % (nf, threads, wall)}
        emit(line)
    bank.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
