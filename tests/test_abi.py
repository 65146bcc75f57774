"""The C-ABI library loads and exports exactly what include/vo_b200.h declares (no compute calls: no GPU here)."""
import ctypes
import os
import re
import shutil
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "vo_b200.h")
LIB = os.path.join(ROOT, "visual-odometry-pipeline_b200", "libvo_b200.so")
# the toolkit's bin/ need not be on PATH; csrc/build.sh finds nvcc under /usr/local/cuda the same way
CUOBJDUMP = shutil.which("cuobjdump") or os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "cuobjdump")


def _declared():
    src = open(HEADER).read()
    return sorted(set(re.findall(r"^VO_API [^;(]*?\b(vo_[a-z0-9_]+)\(", src, flags=re.M)))


def test_header_declares_the_expected_entry_points():
    names = _declared()
    for must in ("vo_create", "vo_destroy", "vo_last_error", "vo_match_u8", "vo_match_f32", "vo_backproject_dense",
                 "vo_gather_backproject", "vo_hypotheses", "vo_pnp_ransac", "vo_pipeline"):
        assert must in names


def test_library_exports_every_declared_symbol_and_nothing_else():
    assert os.path.exists(LIB), "build the library first: python -c 'import __graft_entry__ as g; g.build()'"
    out = subprocess.check_output(["nm", "-D", "--defined-only", LIB], text=True)
    exported = sorted(l.split()[-1] for l in out.splitlines() if " T " in l)
    assert exported == _declared()
    lib = ctypes.CDLL(LIB)
    for name in _declared():
        getattr(lib, name)


def test_binding_prototypes_cover_the_header_and_abi_version():
    import vo_b200
    from vo_b200 import _lib
    assert sorted(_lib.PROTOTYPES) == _declared()
    lib = _lib.load()
    assert lib.vo_abi_version() == _lib.VO_ABI_VERSION
    src = open(HEADER).read()
    for name in ("VO_MODE_RATIO", "VO_MODE_MUTUAL", "VO_MODE_RATIO_MUTUAL", "VO_MODE_THRESH_MUTUAL", "VO_MODE_THRESH",
                 "VO_MODE_NN", "VO_NORM_HAMMING", "VO_NORM_L2_U8", "VO_NORM_HAMMING_TC", "VO_METRIC_L2", "VO_METRIC_COSINE", "VO_PREC_TF32X3",
                 "VO_PREC_TF32X1", "VO_PREC_FP32_SIMT", "VO_PREC_F16X1", "VO_PREC_F16X3", "VO_ST_NO_MODEL", "VO_ST_TOO_FEW_POINTS", "VO_ST_KP_OUT_OF_IMAGE"):
        m = re.search(rf"#define {name} \(?(-?\d+)\)?", src)
        assert m and int(m.group(1)) == getattr(_lib, name), name


def test_sass_is_sm100a_only():
    out = subprocess.run([CUOBJDUMP, "-lelf", LIB], capture_output=True, text=True).stdout
    archs = set(re.findall(r"sm_(\d+a?)", out))
    assert archs == {"100a"}, archs


def test_no_context_without_a_gpu_means_a_loud_error():
    import torch
    if torch.cuda.is_available():
        return
    import pytest
    from vo_b200 import _lib, ops
    with pytest.raises(_lib.VoError):
        ops.context()
