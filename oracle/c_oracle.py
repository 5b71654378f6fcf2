"""ctypes wrapper of oracle/libekf_oracle.so (the C restatement; TEST / BASELINE infrastructure only)."""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_lib = None


def _cpu_tag():
    """The library is built with -march=native, so its name carries a hash of this host's CPU flags."""
    import hashlib
    flags = ""
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("flags"):
                    flags = line
                    break
    except OSError:
        pass
    return hashlib.sha1(flags.encode()).hexdigest()[:10]


def so_name():
    return "libekf_oracle.%s.so" % _cpu_tag()


def load(build=True):
    global _lib
    if _lib is None:
        so = os.path.join(_HERE, so_name())
        if not os.path.exists(so) and build:
            # built in-tree by __graft_entry__.build(); a host with other CPU flags builds its own copy in a temporary
            # directory, because the tree may be read-only at run time
            import tempfile
            so = os.path.join(tempfile.mkdtemp(prefix="ekf_oracle_"), so_name())
            subprocess.run(["make", "-C", _HERE, "SO=" + so], check=True, capture_output=True)
        _lib = C.CDLL(so)
        _lib.ekf_oracle_step_batch.restype = C.c_int
        _lib.ekf_oracle_max_threads.restype = C.c_int
    return _lib


def max_threads():
    return int(load().ekf_oracle_max_threads())


def step_batch(x, P, types, nfeat, zc, has, u, std_a=0.007, std_alpha=0.007, std_z=1.0, delta_t=1.0,
               chi2=5.9915, p_free=0.99, max_hyp=1000, fixed_hyp=0, nthreads=0):
    """In-place reference step on x [B,nmax], P [B,nmax,nmax]; returns (flags [B,N], stats [B,4])."""
    lib = load()
    B, nmax = x.shape
    N = types.shape[1]
    for a, dt in ((x, np.float64), (P, np.float64), (types, np.uint8), (nfeat, np.int32), (zc, np.float64),
                  (has, np.uint8), (u, np.float64)):
        assert a.dtype == dt and a.flags["C_CONTIGUOUS"], (a.dtype, dt)
    assert P.shape == (B, nmax, nmax) and zc.shape == (B, N, 2) and has.shape == (B, N) and u.shape[0] == B
    flags = np.zeros((B, N), dtype=np.uint8)
    stats = np.zeros((B, 4), dtype=np.int32)
    par = np.array([std_a, std_alpha, std_z, delta_t, chi2, p_free, max_hyp, fixed_hyp], dtype=np.float64)
    p = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
    rc = lib.ekf_oracle_step_batch(C.c_int(B), C.c_int(N), C.c_int(nmax), p(x), p(P), p(types), p(nfeat), p(zc), p(has),
                                   p(u), C.c_int(u.shape[1]), p(par), p(flags), p(stats), C.c_int(nthreads))
    assert rc == 0
    return flags, stats
