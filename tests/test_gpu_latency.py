"""Latency path (BASELINE configs[1]: a single filter, N=100, 256 hypotheses per frame): the filter step replayed from
a captured CUDA graph (ekfslam_step_graph) and the thread-block-cluster RANSAC kernel it uses for few filters with a
fixed hypothesis budget.  Both must reproduce the plain path bit for bit."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("B,N,fixed", [(1, 100, 256), (3, 40, 0), (2, 24, 64)])
def test_step_graph_equals_step(B, N, fixed):
    import ekf_slam_b200 as pkg
    import ekf_slam_b200.synth as synth
    frames, n_u = 6, max(64, fixed)
    seq = synth.SynthSequence(B=B, N=N, T=frames, seed=1234, n_u=n_u)
    x0, P0, types = seq.initial_state()
    banks = [pkg.FilterBank(B, N) for _ in range(2)]
    for bk in banks:
        bk.set_params(fixed_hyp=fixed)
        bk.upload_feature_types(types)
        bk.upload_state(x0, P0)
    for t in range(1, frames + 1):
        zc, has, u = seq.frame(t)[0], seq.frame(t)[1], seq.uniforms(t, n_u)
        for g, bk in enumerate(banks):
            bk.upload_candidates(zc, has)
            bk.upload_uniforms(u)
            bk.step(reset=True, match_mode=1, graph=bool(g))
        if t == 3:   # a parameter change invalidates the captured graph (same change on both banks)
            for bk in banks:
                bk.set_params(std_z=1.0, fixed_hyp=fixed)
        xa, Pa, _ = banks[0].download_state()
        xb, Pb, _ = banks[1].download_state()
        assert np.array_equal(xa, xb) and np.array_equal(Pa, Pb), t
        assert np.array_equal(banks[0].download_flags(), banks[1].download_flags()), t
        sa, sb = banks[0].download_stats(), banks[1].download_stats()
        for k in sa:
            assert np.array_equal(sa[k], sb[k]), (t, k)
    # the graph path launched as many kernels as the plain one (counted, not guessed)
    assert banks[0].launch_count == banks[1].launch_count
    for bk in banks:
        bk.close()


def test_cluster_ransac_equals_block_ransac():
    """k_ransac_fixed_cluster (8 CTAs per filter, supports exchanged through distributed shared memory) against
    k_ransac's fixed-budget branch on the same two filters: alone as a batch of 2 they take the cluster kernel, as the
    first two filters of a batch of 64 the block kernel (the cluster kernel needs B * 8 <= 2 * SMs).  SynthSequence seeds
    filter b with seed + b, so both batches start those filters from identical inputs.  Same flags, statistics, state."""
    import ekf_slam_b200 as pkg
    import ekf_slam_b200.synth as synth
    B, N, fixed, frames = 2, 100, 256, 3
    out = []
    for batch in (B, 64):
        seq = synth.SynthSequence(B=batch, N=N, T=frames, seed=4321, n_u=fixed, p_outlier=0.3)
        x0, P0, types = seq.initial_state()
        bank = pkg.FilterBank(batch, N)
        bank.set_params(fixed_hyp=fixed)
        bank.upload_feature_types(types)
        bank.upload_state(x0, P0)
        rec = []
        for t in range(1, frames + 1):
            bank.upload_candidates(*seq.frame(t))
            bank.upload_uniforms(seq.uniforms(t, fixed))
            bank.step()
            rec.append((bank.download_flags(nb=B), bank.download_stats(nb=B), bank.download_state(nb=B, want_P=False)[0]))
        out.append(rec)
        bank.close()
    for (fa, sa, xa), (fb, sb, xb) in zip(*out):
        assert np.array_equal(fa, fb) and np.array_equal(xa, xb)
        for k in sa:
            assert np.array_equal(sa[k], sb[k]), k
        assert (sa["ransac_iters"] == fixed).all() and (sa["max_support"] > 10).all()
