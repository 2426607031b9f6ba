"""CPU: the C-ABI library exists, loads, and exports every symbol include/optb.h declares."""
import ctypes
import os
import re

import pytest

from optable_b200 import _abi as A
from optable_b200 import build

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    src = open(os.path.join(ROOT, "include", "optb.h")).read()
    return sorted(set(re.findall(r"\b(optb_[a-z0-9_]+)\s*\(", src)))


def test_header_and_python_mirror_agree():
    assert sorted(A.EXPORTED_SYMBOLS) == _declared()
    src = open(os.path.join(ROOT, "include", "optb.h")).read()
    assert f"#define OPTB_ABI_VERSION {A.ABI_VERSION}" in src
    for name, val in (("OPTB_NI_STRIDE", A.NI_STRIDE), ("OPTB_NF_STRIDE", A.NF_STRIDE), ("OPTB_MON_STRIDE", A.MON_STRIDE),
                      ("OPTB_NF_CAPMAX", A.NF_CAPMAX), ("OPTB_POLY_HEADER", A.POLY_HEADER), ("OPTB_C_COUNT", A.C_COUNT)):
        assert re.search(rf"{name}\s*=\s*{val}\b", src), name
    # optb_trace_plan's variant bits
    plan = {m[0]: int(m[1]) for m in re.findall(r"#define OPTB_(PLAN_\w+)\s+\(1u << (\d+)\)", src)}
    assert len(plan) == 9
    for name, shift in plan.items():
        assert getattr(A, name) == 1 << shift, name
    assert re.search(rf"#define OPTB_PLAN_BOX_SHIFT\s+{A.PLAN_BOX_SHIFT}\b", src)
    assert re.search(r"#define OPTB_PLAN_BOX_MASK\s+\(3u << OPTB_PLAN_BOX_SHIFT\)", src) and A.PLAN_BOX_MASK == 3 << A.PLAN_BOX_SHIFT


def test_library_exports_all_symbols():
    so = build.build_extension()
    L = ctypes.CDLL(so)
    for sym in _declared():
        assert hasattr(L, sym), sym
    L.optb_abi_version.restype = ctypes.c_int
    assert L.optb_abi_version() == A.ABI_VERSION


def test_struct_sizes():
    assert ctypes.sizeof(A.SceneDesc) == 6 * 4 + 8 + 6 * 8
    assert ctypes.sizeof(A.Rays) == 8 + 15 * 8 + 8
    assert ctypes.sizeof(A.Params) == 8 + 8 + 10 * 4
    assert ctypes.sizeof(A.Result) == 2 * 8 + (13 + 3 + 1 + 1 + 2 + 10 + 2) * 8 + 4 * 8


def test_product_fails_loudly_without_gpu_or_library(monkeypatch, tmp_path):
    """No CPU fallback: without a CUDA device the engine raises; without the shared library the loader raises."""
    import pytest
    import torch

    from optable_b200 import backend

    if not torch.cuda.is_available():
        with pytest.raises(backend.BackendError):
            backend.Engine.get(0)
        import optable_b200 as ob

        table = ob.OpticalTable()
        table.add_components([ob.Mirror([0, 0, 0])])
        with pytest.raises(backend.BackendError):
            table.ray_tracing([ob.Ray([-1, 0, 0], [1, 0, 0])])
    monkeypatch.setattr(backend, "_lib", None)
    monkeypatch.setattr(backend, "_SO", str(tmp_path / "missing.so"))
    with pytest.raises(backend.BackendError):
        backend.lib()


def test_product_never_imports_the_oracle():
    """The checker is test infrastructure: nothing under optable_b200/ may reference it."""
    import glob

    for path in glob.glob(os.path.join(ROOT, "optable_b200", "**", "*"), recursive=True):
        if os.path.isfile(path) and path.endswith((".py", ".cu", ".cuh", ".h")):
            text = open(path).read()
            assert "import oracle" not in text and "from oracle" not in text and "optb_oracle" not in text, path


def _build_c_demo(tmp_path):
    import shutil
    import subprocess

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("gcc not available")
    libdir = os.path.join(root, "optable_b200")
    exe = str(tmp_path / "optb_demo")
    subprocess.run([gcc, "-std=c99", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(root, "include"),
                    os.path.join(root, "examples", "optb_demo.c"), "-L", libdir, "-loptb", "-lm", f"-Wl,-rpath,{libdir}", "-o", exe],
                   check=True)
    return exe


def test_header_is_plain_c_and_a_c_program_links(tmp_path):
    """include/optb.h compiles as C99 (no C++ or torch types on the boundary) and examples/optb_demo.c, a host
    program written against nothing but that header, links with liboptb.so. Without a GPU it must stop at
    optb_ctx_create with an error, not fall back to anything."""
    import subprocess

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    subprocess.run(["gcc", "-std=c99", "-pedantic", "-Wall", "-Werror", "-fsyntax-only", "-x", "c",
                    os.path.join(root, "include", "optb.h")], check=True)
    exe = _build_c_demo(tmp_path)
    import torch

    if not torch.cuda.is_available():
        run = subprocess.run([exe], capture_output=True, text=True)
        assert run.returncode == 1 and "optb_ctx_create" in run.stderr


@pytest.mark.gpu
def test_c_demo_runs_on_the_device(tmp_path):
    """The same C program end to end on the GPU: 4 rays, a splitting mirror, one monitor; it checks its own rows."""
    import subprocess

    run = subprocess.run([_build_c_demo(tmp_path)], capture_output=True, text=True)
    assert run.returncode == 0 and run.stdout.strip().endswith("OK"), run.stdout + run.stderr
    assert "segments 12 interactions 4 monitor_rows 4 status 0" in run.stdout
