"""CPU checks of the drop-in boundary: the C-ABI library loads, exports every symbol include/*.h declares,
rejects bad arguments without touching a GPU, and the product never reaches into oracle/."""
import ctypes as C
import os
import re
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "d3d_b200", "libd3d_b200.so")


def _declared():
    src = open(os.path.join(ROOT, "include", "d3d_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(d3d_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    assert os.path.exists(LIB), "run __graft_entry__.build() first"
    lib = C.CDLL(LIB)
    names = _declared()
    assert len(names) >= 40
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/d3d_b200.h but not exported"
    lib.d3d_abi_version.restype = C.c_int
    assert lib.d3d_abi_version() == 5
    lib.d3d_error_string.restype = C.c_char_p
    assert lib.d3d_error_string(3) == b"workspace too small"


def test_argument_validation_without_gpu():
    """Error paths return codes before any CUDA call, so they are checkable on a CPU-only box."""
    lib = C.CDLL(LIB)
    i64, vp = C.c_int64, C.c_void_p
    # negative sizes / ld < m -> invalid argument
    assert lib.d3d_iou2dr_f32(vp(0), i64(-1), vp(0), i64(2), vp(0), i64(2), vp(0), C.c_size_t(0), vp(0)) == 1
    assert lib.d3d_iou2dr_f32(vp(8), i64(2), vp(8), i64(4), vp(8), i64(3), vp(0), C.c_size_t(0), vp(0)) == 1
    # empty problem is a no-op
    assert lib.d3d_iou2dr_f64(vp(0), i64(0), vp(0), i64(5), vp(0), i64(5), vp(0), C.c_size_t(0), vp(0)) == 0
    # workspace too small
    assert lib.d3d_iou2dr_f32(vp(8), i64(2), vp(8), i64(2), vp(8), i64(2), vp(8), C.c_size_t(16), vp(0)) == 3
    # NMS: unsupported iou type (reference "Unsupported iou type!"), unknown supression type
    nms = lib.d3d_nms2d_f32
    nms.argtypes = [vp, vp, i64, C.c_int, C.c_int, C.c_float, C.c_float, C.c_float, vp, vp, C.c_size_t, vp]
    assert nms(8, 8, 4, 4, 0, 0.5, 0, 0, 8, 8, 1 << 30, 0) == 1
    assert nms(8, 8, 4, 2, 3, 0.5, 0, 0, 8, 8, 1 << 30, 0) == 1   # supression types are HARD / LINEAR / GAUSSIAN
    lib.d3d_iou_workspace_bytes.restype = C.c_size_t
    lib.d3d_iou_workspace_bytes.argtypes = [i64, i64, C.c_int]
    assert lib.d3d_iou_workspace_bytes(1000, 1000, 0) >= 2 * 1000 * 32
    # scatter: bad align / dim
    dims = (C.c_int64 * 3)(4, 4, 4)
    sc = lib.d3d_aligned_scatter_forward
    sc.argtypes = [vp, i64, C.c_int32, vp, i64, i64, C.POINTER(C.c_int64), C.c_int, C.c_int, vp, vp]
    assert sc(8, 1, 2, 8, 1, 1, dims, 0, 0, 8, 0) == 1   # DROP is not a kernel mode
    assert sc(8, 1, 4, 8, 1, 1, dims, 1, 0, 8, 0) == 1   # dim 4


def test_tuning_knob_table():
    """d3d_tuning_set accepts the knobs that force a path some input reaches on its own (plus NMS_STOP, the phase timing of bench.py)
    and rejects the names of retired knobs with INVALID_ARGUMENT."""
    lib = C.CDLL(LIB)
    lib.d3d_tuning_set.argtypes = [C.c_char_p, C.c_int, C.c_int]
    kept = ["NMS_PATH", "NMS_FIX", "NMS_BATCH_PATH", "SORT_COOP", "CROP_PATH", "SCATTER_PATH", "VOX_ROUTE", "NMS_STOP"]
    retired = ["NMS_NT", "NMS_STAGE", "VOX_CLUSTER", "VOX_MAXCL", "VOX_CF", "VOX_ROLES"]
    try:
        for k in kept:
            assert lib.d3d_tuning_set(b"D3D_B200_" + k.encode(), 0, 1) == 0, k
        for k in retired:
            assert lib.d3d_tuning_set(b"D3D_B200_" + k.encode(), 0, 1) == 1, k
    finally:
        for k in kept:
            lib.d3d_tuning_set(b"D3D_B200_" + k.encode(), 0, 0)


def test_product_never_touches_the_oracle():
    """The oracle is test infrastructure: nothing under d3d_b200/ may import, link or open it."""
    bad = []
    for dp, _, files in os.walk(os.path.join(ROOT, "d3d_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cpp", "Makefile")):
                txt = open(os.path.join(dp, f), errors="ignore").read()
                if re.search(r"\boracle\b|d3d_oracle|host_twin|libtwin", txt):
                    bad.append(os.path.join(dp, f))
    assert not bad, bad
    out = subprocess.run(["ldd", LIB], capture_output=True, text=True).stdout
    assert "oracle" not in out and "twin" not in out


def test_sass_is_sm100a_only():
    out = subprocess.run(["cuobjdump", "-lelf", LIB], capture_output=True, text=True).stdout
    archs = set(re.findall(r"sm_(\d+a?)", out))
    assert archs == {"100a"}, archs


def test_import_fails_loudly_without_extension(tmp_path):
    """No CPU fallback: importing the package without the built library raises ImportError."""
    import shutil
    dst = tmp_path / "d3d_b200"
    shutil.copytree(os.path.join(ROOT, "d3d_b200"), dst, ignore=shutil.ignore_patterns("*.so", "*.o", "csrc", "__pycache__"))
    r = subprocess.run([sys.executable, "-c", "import d3d_b200"], cwd=tmp_path, capture_output=True, text=True)
    assert r.returncode != 0 and "ImportError" in r.stderr
