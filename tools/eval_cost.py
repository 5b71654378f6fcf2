"""Cost of scoring the filters against the ground truth (ekfslam_evaluate) at the bench shape.

B=4096 filters x N=100 features on a SynthSequence (bench.py's default seed), frame-0 maps built on the device as
bench.py builds them, the sequence's own truth uploaded as the world (SynthSequence.truth_world(), tags = feature index).
After a warm-up, windows of K device-resident steps with and without one evaluate(t) per step alternate (CUDA events
around each window); a separate window with per-kernel timing on gives the k_eval slot's time per launch.  Prints one
JSON line with the card name and power limit read in the same run (nvidia-smi, read-only query).

    python tools/eval_cost.py [--batch 4096 --features 100 --steps 8 --reps 3 --warmup 4] [--out FILE]
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--features", type=int, default=100)
    ap.add_argument("--steps", type=int, default=8, help="steps per timed window")
    ap.add_argument("--reps", type=int, default=3, help="pairs of windows (with / without evaluation)")
    ap.add_argument("--warmup", type=int, default=4)
    ap.add_argument("--seed", type=int, default=2024)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()

    import torch
    import ekf_slam_b200 as pkg
    import ekf_slam_b200.synth as synth

    if not torch.cuda.is_available():
        raise SystemExit("eval_cost.py needs a CUDA device (there is no CPU fallback)")
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
    bank.upload_feature_meta(tag=np.tile(np.arange(N, dtype=np.int32), (B, 1)))
    bank.world_upload(seq.truth_world())
    zc_dev = torch.from_numpy(seq.zc).to(dev)
    fl_dev = torch.from_numpy((seq.has * pkg.F_CAND).astype(np.uint8)).to(dev)
    u_dev = torch.from_numpy(np.ascontiguousarray(np.transpose(seq.U, (1, 0, 2)))).to(dev)
    torch.cuda.synchronize(dev)

    def window(t0, evaluate):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for t in range(t0, t0 + K):
            bank.bind_frame(zc_dev[t].data_ptr(), fl_dev[t].data_ptr(), u_dev[t].data_ptr(), n_u)
            bank.step(reset=True, match_mode=1)
            if evaluate:
                bank.evaluate(t)
        e1.record(stream)
        torch.cuda.synchronize(dev)
        return e0.elapsed_time(e1) / K

    t = 1
    for _ in range(W):   # warm-up: every kernel of the step and k_eval
        bank.bind_frame(zc_dev[t].data_ptr(), fl_dev[t].data_ptr(), u_dev[t].data_ptr(), n_u)
        bank.step(reset=True, match_mode=1)
        bank.evaluate(t)
        t += 1
    torch.cuda.synchronize(dev)
    with_ms, without_ms = [], []
    for r in range(R):   # alternate, and alternate which arm goes first
        for ev in ((True, False) if r % 2 == 0 else (False, True)):
            (with_ms if ev else without_ms).append(window(t, ev))
            t += K
    bank.enable_timing(True)
    window(t, True)
    kt = bank.kernel_times()
    bank.enable_timing(False)
    bank.unbind_frame()
    ev_ms, ev_n = kt["k_eval"]
    step_kernels_ms = sum(ms for name, (ms, n) in kt.items() if name != "k_eval") / K
    tot = bank.download_eval(totals=True)
    res = dict(
        tool="eval_cost", card=card(), B=B, N=N, steps_per_window=K, windows_per_arm=R,
        step_ms_without_eval=without_ms, step_ms_with_eval=with_ms,
        step_ms_without_eval_median=float(np.median(without_ms)), step_ms_with_eval_median=float(np.median(with_ms)),
        k_eval_ms_per_launch=ev_ms / max(ev_n, 1), k_eval_launches=ev_n,
        k_eval_fraction_of_step=(ev_ms / max(ev_n, 1)) / float(np.median(without_ms)),
        step_kernel_ms_timed_window=step_kernels_ms,
        frames_scored=int(tot["frames"][0]), mean_camera_nees_pose=float(np.nanmean(tot["nees_pose"] / tot["frames"])),
        mean_map_nees_per_feature=float(tot["map_nees"].sum() / max(tot["n_map"].sum(), 1)))
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")
    bank.close()


if __name__ == "__main__":
    main()
