"""N>1 host logic on CPU: world_size-2 gloo processes gather their shards' evaluation records
(sharding.gather_eval) into float64 arrays in global filter order."""
import os
import socket

import numpy as np
import torch.distributed as dist
import torch.multiprocessing as mp

import ekf_slam_b200.sharding as sharding
from ekf_slam_b200._lib import EVAL_FIELDS


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _records(b0, nb):
    """Stand-in records: deterministic functions of the global filter index, with the dtypes of download_eval()."""
    g = np.arange(b0, b0 + nb)
    rec = {k: (g + 0.25) * (i + 1) / 3.0 for i, k in enumerate(EVAL_FIELDS[:6])}
    rec.update(n_map=(g * 3).astype(np.int32), n_skip=(g % 4).astype(np.int32),
               frames=np.full(nb, 5, dtype=np.int32), status=(g % 8).astype(np.int32))
    return rec


def _worker(rank, world, port, B, out_dir):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        b0, nb = sharding.partition(B, world, rank)
        allrec = sharding.gather_eval(_records(b0, nb), n_filters_total=B)
        np.savez(os.path.join(out_dir, "r%d.npz" % rank), **allrec)
    finally:
        dist.destroy_process_group()


def test_two_rank_gloo_gather_eval(tmp_path):
    B, world = 7, 2
    port = _free_port()
    mp.spawn(_worker, args=(world, port, B, str(tmp_path)), nprocs=world, join=True)
    full = _records(0, B)
    r0 = np.load(tmp_path / "r0.npz")
    r1 = np.load(tmp_path / "r1.npz")
    for k in EVAL_FIELDS:
        assert r0[k].dtype == np.float64 and r0[k].shape == (B,)
        assert np.array_equal(r0[k], r1[k])
        assert np.array_equal(r0[k], np.asarray(full[k], dtype=np.float64)), k


def test_single_process_gather_eval_is_the_local_records():
    rec = _records(0, 3)
    out = sharding.gather_eval(rec)
    for k in EVAL_FIELDS:
        assert out[k].dtype == np.float64 and np.array_equal(out[k], np.asarray(rec[k], dtype=np.float64))
