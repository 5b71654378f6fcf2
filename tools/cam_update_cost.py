"""Cost of the camera-state measurement update (ekfslam_update_camera) at the bench shape.

B=4096 filters x N=100 features on a SynthSequence (bench.py's default seed), frame-0 maps built on the device as
bench.py builds them.  After every step each filter gets an m=3 position fix (which=0) from the sequence's true pose.
After a warm-up, windows of K device-resident steps with and without the fix alternate (CUDA events around each window);
a separate window with per-kernel timing on gives the time per launch of the two new slots, k_cam_update and
k_downdate_cam.  The downdate's roofline share is the bytes it must move (P read and written once: 2 n^2 8 bytes per
filter at the mean state size) over its time, as a share of the HBM rate tools/microbench_fp64 measures in the same run
(or of the 7.7 TB/s data-sheet figure when that binary is missing).  Prints one JSON line with the card name and power
limit read in the same run (nvidia-smi, read-only query).

    python tools/cam_update_cost.py [--batch 4096 --features 100 --steps 8 --reps 3 --warmup 4] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv"], capture_output=True,
                           text=True, timeout=60)
        return r.stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        return "nvidia-smi unavailable: %s" % e


def hbm_peak_gbs():
    """Measured HBM rate (GB/s) from tools/microbench_fp64 (built by __graft_entry__.build()), or None."""
    exe = os.path.join(ROOT, "tools", "microbench_fp64")
    if not os.path.exists(exe):
        return None
    try:
        out = subprocess.run([exe], capture_output=True, text=True, timeout=300).stdout
    except (OSError, subprocess.SubprocessError):
        return None
    for line in out.splitlines():
        try:
            d = json.loads(line)
        except ValueError:
            continue
        if isinstance(d, dict) and "copy_gbs" in d:
            return float(d["copy_gbs"])
    return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--features", type=int, default=100)
    ap.add_argument("--steps", type=int, default=8, help="steps per timed window")
    ap.add_argument("--reps", type=int, default=3, help="pairs of windows (with / without the fix)")
    ap.add_argument("--warmup", type=int, default=4)
    ap.add_argument("--seed", type=int, default=2024)
    ap.add_argument("--sigma", type=float, default=0.01, help="std of the position fix")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()

    import torch
    import ekf_slam_b200 as pkg
    import ekf_slam_b200.synth as synth

    if not torch.cuda.is_available():
        raise SystemExit("cam_update_cost.py needs a CUDA device (there is no CPU fallback)")
    B, N, K, W, R = args.batch, args.features, args.steps, args.warmup, args.reps
    n_u = 64
    T = W + 2 * R * K + K
    dev = torch.device("cuda", 0)
    seq = synth.SynthSequence(B=B, N=N, T=T, seed=args.seed, n_u=n_u)
    bank = pkg.FilterBank(B, N, device=0)
    stream = torch.cuda.Stream(dev)
    torch.cuda.set_stream(stream)
    bank.set_stream(stream.cuda_stream)
    bank.reset_filters()
    for k in range(N):
        bank.add_features_inverse_depth(np.ascontiguousarray(seq.zc[0, :, k]))
    zc_dev = torch.from_numpy(seq.zc).to(dev)
    fl_dev = torch.from_numpy((seq.has * pkg.F_CAND).astype(np.uint8)).to(dev)
    u_dev = torch.from_numpy(np.ascontiguousarray(np.transpose(seq.U, (1, 0, 2)))).to(dev)
    H = np.zeros((3, 13))
    H[:, :3] = np.eye(3)
    Rm = args.sigma ** 2 * np.eye(3)
    rng = np.random.RandomState(args.seed)
    # the fixes of every frame are drawn up front, so no host work sits inside a timed window
    fixes = [np.ascontiguousarray(seq.pose_r[:, t] + args.sigma * rng.standard_normal((B, 3))) for t in range(T + 1)]
    torch.cuda.synchronize(dev)

    def window(t0, fix):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for t in range(t0, t0 + K):
            bank.bind_frame(zc_dev[t].data_ptr(), fl_dev[t].data_ptr(), u_dev[t].data_ptr(), n_u)
            bank.step(reset=True, match_mode=1)
            if fix:
                bank.update_camera(H, fixes[t], Rm, which=0)
        e1.record(stream)
        torch.cuda.synchronize(dev)
        return e0.elapsed_time(e1) / K

    t = 1
    for _ in range(W):   # warm-up: every kernel of the step and of the fix
        bank.bind_frame(zc_dev[t].data_ptr(), fl_dev[t].data_ptr(), u_dev[t].data_ptr(), n_u)
        bank.step(reset=True, match_mode=1)
        bank.update_camera(H, fixes[t], Rm, which=0)
        t += 1
    torch.cuda.synchronize(dev)
    with_ms, without_ms = [], []
    for r in range(R):   # alternate, and alternate which arm goes first
        for fx in ((True, False) if r % 2 == 0 else (False, True)):
            (with_ms if fx else without_ms).append(window(t, fx))
            t += K
    bank.enable_timing(True)
    window(t, True)
    kt = bank.kernel_times()
    bank.enable_timing(False)
    bank.unbind_frame()
    cu_ms, cu_n = kt["k_cam_update"]
    dd_ms, dd_n = kt["k_downdate_cam"]
    st = bank.download_camera_update()
    _, _, ns = bank.download_state(want_P=False)
    n_mean = float(ns.mean())
    p_bytes = float(np.sum(2.0 * ns.astype(np.float64) ** 2 * 8))   # P read + written once, lower+upper as stored
    dd_per = dd_ms / max(dd_n, 1)
    peak = hbm_peak_gbs()
    peak_src = "tools/microbench_fp64" if peak else "data sheet (7.7 TB/s)"
    peak = peak or 7700.0
    gbs = p_bytes / (dd_per * 1e-3) / 1e9
    res = dict(
        tool="cam_update_cost", card=card(), B=B, N=N, m=3, mean_state_size=n_mean, steps_per_window=K,
        windows_per_arm=R, step_ms_without_fix=without_ms, step_ms_with_fix=with_ms,
        step_ms_without_fix_median=float(np.median(without_ms)), step_ms_with_fix_median=float(np.median(with_ms)),
        fix_ms_per_call_median=float(np.median(with_ms) - np.median(without_ms)),
        k_cam_update_ms_per_launch=cu_ms / max(cu_n, 1), k_downdate_cam_ms_per_launch=dd_per, launches=cu_n,
        downdate_p_bytes=p_bytes, downdate_gbs=gbs, hbm_peak_gbs=peak, hbm_peak_source=peak_src,
        downdate_share_of_hbm_peak=gbs / peak, applied=int((st["status"] == 0).sum()),
        mean_nis_last_fix=float(np.nanmean(st["nis"])))
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")
    bank.close()


if __name__ == "__main__":
    main()
