"""Cost of the known-landmark update (ekfslam_update_landmarks) at the bench shape.

B=4096 filters x N=100 features on a SynthSequence (bench.py's default seed), frame-0 maps built on the device as
bench.py builds them.  Every filter has 6 landmarks, world points 0..5 of its sequence at their true positions; after
every step the device world (the sequence's own truth, ekfslam_world_upload) draws their observations
(ekfslam_world_landmark_obs) and one update (which=0, 0.5 px, chi-square gate 5.9915) follows.  After a warm-up,
windows of K device-resident steps with and without the update alternate (CUDA events around each window); a separate
window with per-kernel timing on gives the time per launch of the two new slots, k_lm_update and k_downdate_lm.  The
downdate's roofline share is the bytes it must move (P read and written once: 2 n^2 8 bytes per filter at the mean
state size, over the filters the last update applied to) over its time, as a share of the HBM rate tools/microbench_fp64 measures in the same run (or of the
7.7 TB/s data-sheet figure when that binary is missing).  Prints one JSON line with the card name and power limit read
in the same run (nvidia-smi, read-only query).

    python tools/landmark_update_cost.py [--batch 4096 --features 100 --steps 8 --reps 3 --warmup 4] [--out FILE]
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
    ap.add_argument("--landmarks", type=int, default=6)
    ap.add_argument("--steps", type=int, default=8, help="steps per timed window")
    ap.add_argument("--reps", type=int, default=3, help="pairs of windows (with / without the update)")
    ap.add_argument("--warmup", type=int, default=4)
    ap.add_argument("--seed", type=int, default=2024)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()

    import torch
    import ekf_slam_b200 as pkg
    import ekf_slam_b200.synth as synth

    if not torch.cuda.is_available():
        raise SystemExit("landmark_update_cost.py needs a CUDA device (there is no CPU fallback)")
    B, N, Lm, K, W, R = args.batch, args.features, args.landmarks, args.steps, args.warmup, args.reps
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
    bank.world_upload(seq.truth_world())
    bank.upload_landmarks(seq.points[:, :Lm], tag=np.tile(np.arange(Lm, dtype=np.int32), (B, 1)))
    zc_dev = torch.from_numpy(seq.zc).to(dev)
    fl_dev = torch.from_numpy((seq.has * pkg.F_CAND).astype(np.uint8)).to(dev)
    u_dev = torch.from_numpy(np.ascontiguousarray(np.transpose(seq.U, (1, 0, 2)))).to(dev)
    gate = 5.9915
    torch.cuda.synchronize(dev)

    def window(t0, upd):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for t in range(t0, t0 + K):
            bank.bind_frame(zc_dev[t].data_ptr(), fl_dev[t].data_ptr(), u_dev[t].data_ptr(), n_u)
            bank.step(reset=True, match_mode=1)
            if upd:
                bank.world_landmark_obs(t)
                bank.update_landmarks(seq.noise_px, gate=gate, which=0)
        e1.record(stream)
        torch.cuda.synchronize(dev)
        return e0.elapsed_time(e1) / K

    t = 1
    for _ in range(W):   # warm-up: every kernel of the step and of the update
        bank.bind_frame(zc_dev[t].data_ptr(), fl_dev[t].data_ptr(), u_dev[t].data_ptr(), n_u)
        bank.step(reset=True, match_mode=1)
        bank.world_landmark_obs(t)
        bank.update_landmarks(seq.noise_px, gate=gate, which=0)
        t += 1
    torch.cuda.synchronize(dev)
    with_ms, without_ms = [], []
    for r in range(R):   # alternate, and alternate which arm goes first
        for up in ((True, False) if r % 2 == 0 else (False, True)):
            (with_ms if up else without_ms).append(window(t, up))
            t += K
    bank.enable_timing(True)
    window(t, True)
    kt = bank.kernel_times()
    bank.enable_timing(False)
    bank.unbind_frame()
    lu_ms, lu_n = kt["k_lm_update"]
    dd_ms, dd_n = kt["k_downdate_lm"]
    st = bank.download_landmark_update()
    _, _, ns = bank.download_state(want_P=False)
    n_mean = float(ns.mean())
    upd = st["status"] == pkg.LMU_APPLIED          # the downdate skips filters that were not updated (ktot = 0)
    p_bytes = float(np.sum(2.0 * ns[upd].astype(np.float64) ** 2 * 8))   # P read + written once, lower+upper as stored
    dd_per = dd_ms / max(dd_n, 1)
    peak = hbm_peak_gbs()
    peak_src = "tools/microbench_fp64" if peak else "data sheet (7.7 TB/s)"
    peak = peak or 7700.0
    gbs = p_bytes / (dd_per * 1e-3) / 1e9
    res = dict(
        tool="landmark_update_cost", card=card(), B=B, N=N, landmarks=Lm, mean_state_size=n_mean,
        steps_per_window=K, windows_per_arm=R, step_ms_without_update=without_ms, step_ms_with_update=with_ms,
        step_ms_without_update_median=float(np.median(without_ms)),
        step_ms_with_update_median=float(np.median(with_ms)),
        update_ms_per_call_median=float(np.median(with_ms) - np.median(without_ms)),
        k_lm_update_ms_per_launch=lu_ms / max(lu_n, 1), k_downdate_lm_ms_per_launch=dd_per, launches=lu_n,
        downdate_p_bytes=p_bytes, downdate_gbs=gbs, hbm_peak_gbs=peak, hbm_peak_source=peak_src,
        downdate_share_of_hbm_peak=gbs / peak, applied=int((st["status"] == pkg.LMU_APPLIED).sum()),
        mean_k=float(st["k"].mean()), mean_nis_last_update=float(np.nanmean(st["nis"])))
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")
    bank.close()


if __name__ == "__main__":
    main()
