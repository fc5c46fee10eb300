"""Host-side checks that need no GPU: the C-ABI library builds for sm_100a, loads, exports every symbol the
header declares, and fails loudly (no CPU fallback) when there is no CUDA device."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as g
    path = g.build_engine()
    return ctypes.CDLL(path)


def test_exports_every_declared_symbol(lib):
    hdr = open(os.path.join(ROOT, "include", "loro_b200.h")).read()
    names = set(re.findall(r"\b(lb_[a-z_]+)\s*\(", hdr))
    assert {"lb_import_batch", "lb_import_batch_device", "lb_doc_status", "lb_doc_json", "lb_doc_vv",
            "lb_batch_counters", "lb_batch_timings", "lb_batch_free", "lb_doc_count", "lb_last_error",
            "lb_doc_frontiers", "lb_doc_export_updates", "lb_docset_new", "lb_docset_import", "lb_docset_free"} <= names
    for n in names:
        assert hasattr(lib, n), n


def test_no_cpu_fallback_without_a_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("CUDA device present")
    import loro_b200
    with pytest.raises(loro_b200.EngineUnavailable):
        loro_b200.import_batch([b"loro" + bytes(30)])
    with pytest.raises(loro_b200.EngineUnavailable):
        loro_b200.DocSet()


def test_sass_is_sm100a(lib):
    import shutil
    import subprocess
    import loro_b200
    # the toolkit that build() compiles with, also when its bin/ is not on PATH
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cuobjdump = shutil.which("cuobjdump") or os.path.join(os.path.dirname(nvcc), "cuobjdump")
    out = subprocess.run([cuobjdump, "-lelf", loro_b200.library_path()], capture_output=True, text=True).stdout
    assert "sm_100a" in out, out


def test_library_shares_no_state_with_other_builds_in_the_process(lib):
    """The library defines no GNU-unique symbol of its own: the dynamic loader binds such a symbol to the first library
    of the process that defines it, so a second build of the engine (the emulated one, loaded first when this suite runs
    in one process) would hand the CUDA library its host staging ring."""
    import subprocess
    import loro_b200
    out = subprocess.run(["nm", "-DC", "--defined-only", loro_b200.library_path()], capture_output=True, text=True,
                         check=True).stdout
    unique = [ln for ln in out.splitlines() if ln.split()[1:2] == ["u"] and " std::" not in ln]
    assert not unique, unique


def test_plain_c_caller_compiles_links_and_fails_loudly_without_a_device(lib, tmp_path):
    """include/loro_b200.h is plain C (no torch / C++ types in the signatures): examples/c/import_and_docset.c builds
    with -std=c99 -Wall -Wextra -Werror, links against the library and, without a CUDA device, gets LB_ERR_NO_DEVICE."""
    import subprocess
    import loro_b200
    exe = str(tmp_path / "demo")
    libdir = os.path.dirname(loro_b200.library_path())
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Wextra", "-Werror", "-I" + os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "examples", "c", "import_and_docset.c"), "-L" + libdir, "-lloro_b200", "-o", exe])
    import torch
    if torch.cuda.is_available():
        return
    out = subprocess.run([exe, os.path.join(ROOT, "tests", "golden", "gv1_update.bin")], capture_output=True, text=True,
                         env=dict(os.environ, LD_LIBRARY_PATH=libdir))
    assert out.returncode == 1 and "no CUDA device" in out.stderr, (out.returncode, out.stderr)
