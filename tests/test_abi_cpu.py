"""No-GPU checks of the C-ABI library: it loads, exports every symbol include/ekfslam.h
declares, and fails loudly (no CPU fallback) when there is no device."""
import ctypes as C
import os
import re
import subprocess
import sys

from ekf_slam_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_symbols():
    src = open(os.path.join(ROOT, "include", "ekfslam.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(ekfslam_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    lib = _lib.load()
    syms = _header_symbols()
    assert len(syms) >= 40
    for s in syms:
        assert hasattr(lib, s), "libekfslam.so does not export %s" % s


def test_ctypes_binding_covers_the_header():
    assert sorted(_lib.EXPORTS) == _header_symbols()


def test_defaults_match_reference_constants():
    lib = _lib.load()
    cam = _lib.Camera()
    lib.ekfslam_default_camera(C.byref(cam))
    assert cam.nRows == 240 and cam.nCols == 320
    assert abs(cam.Cx - 1.7945 / 0.0112) < 1e-12 and abs(cam.f - 2.1735) < 1e-15
    p = _lib.Params()
    lib.ekfslam_default_params(C.byref(p))
    assert (p.std_a, p.std_alpha, p.std_z, p.delta_t) == (0.007, 0.007, 1.0, 1.0)
    assert p.chi2_gate == 5.9915 and p.max_hyp == 1000 and p.fixed_hyp == 0 and p.p_spurious_free == 0.99


def test_no_cpu_fallback():
    """Runs in a child process with every device hidden, so that it also checks this where a GPU is present."""
    code = ("import ekf_slam_b200 as pkg\n"
            "try:\n"
            "    pkg.FilterBank(2, 4)\n"
            "except pkg.EkfSlamError as e:\n"
            "    print(e.code, e)\n")
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=ROOT,
                       env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert r.returncode == 0, r.stderr
    code, _, msg = r.stdout.strip().partition(" ")
    assert code == "-5" and "no CPU fallback" in msg, r.stdout


def test_argument_validation_without_device():
    lib = _lib.load()
    h = C.c_void_p()
    assert lib.ekfslam_create(C.byref(h), 0, 0, 4, 37) == -1
    assert b"must be" in lib.ekfslam_last_error()
    assert lib.ekfslam_create(C.byref(h), 0, 1, 4, 12) == -1
    assert lib.ekfslam_synchronize(None) == -1
