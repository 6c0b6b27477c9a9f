"""The C-ABI library builds, loads and exports every entry point include/helmholtz_b200.h declares; the ctypes
table of the Python host layer covers the same set; without a CUDA device the product path fails loudly.
No compute call is made here (CPU container)."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "helmholtz_b200.h")


def declared_functions():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(hp_[a-z0-9_]+)\s*\(", src)))


@pytest.fixture(scope="module")
def libpath():
    from helmholtz_preconditioner_b200 import build
    return build.build()          # no-op when the in-tree .so is newer than its sources


def test_header_declares_the_path():
    names = declared_functions()
    for must in ("hp_create", "hp_assemble_csr", "hp_stencil_matvec", "hp_precond_setup", "hp_precond_apply",
                 "hp_sweep_forward", "hp_sweep_backward", "hp_front_begin", "hp_front_end", "hp_dotc", "hp_mgs"):
        assert must in names


def test_library_exports_every_declared_symbol(libpath):
    lib = ctypes.CDLL(libpath)
    missing = [n for n in declared_functions() if not hasattr(lib, n)]
    assert not missing, missing


def test_ctypes_table_matches_header(libpath):
    from helmholtz_preconditioner_b200 import _lib
    declared = set(declared_functions())
    bound = set(_lib.SIGNATURES)
    assert bound <= declared | {"hp_debug_phases"}, bound - declared
    assert declared - bound == set(), declared - bound
    _lib.load()


def test_no_cpu_fallback(libpath):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    import helmholtz_preconditioner_b200 as hp
    with pytest.raises(hp.HelmholtzB200Error):
        hp.run_solver(20, 5, 3, 30, 2)
    lib = hp.load()
    assert lib.hp_device_ok() == 0
    h = ctypes.c_void_p()
    import numpy as np
    c = np.ones((22, 22))
    assert lib.hp_create(ctypes.byref(h), 20, 5, 1.0, 2.0, 30.0, c.ctypes.data, 0, None) != 0
    assert b"no CUDA device" in lib.hp_last_error()


def test_product_does_not_import_oracle():
    pkg = os.path.join(ROOT, "helmholtz_preconditioner_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in txt and "from oracle" not in txt and "helmholtz_oracle" not in txt, f


def test_sweep_abort_raises_both_flags(tmp_path):
    """hp_raise_abort (csrc/hp_sweep_common.cuh), which a sweep CTA calls when its wait for exchange data runs into
    HP_SPIN_LIMIT, must store the per-launch flag that stops the other CTAs and the sticky flag that hp_sweep_status
    reports, and return.  Compiled for sm_100a: straight-line code with exactly two atomic exchanges and no call (a
    function that calls itself compiles to a CALL into an endless loop, and the stalled sweep would then never end)."""
    import shutil
    import subprocess
    cuda_bin = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin")
    nvcc = shutil.which("nvcc") or shutil.which("nvcc", path=cuda_bin)
    cuobjdump = shutil.which("cuobjdump") or shutil.which("cuobjdump", path=cuda_bin)
    if not nvcc or not cuobjdump:
        pytest.skip("nvcc / cuobjdump not found")
    src = tmp_path / "probe.cu"
    src.write_text('#include "hp_sweep_common.cuh"\n'
                   "__global__ void probe(unsigned int* flag) { hp_raise_abort(flag); }\n")
    cubin = tmp_path / "probe.cubin"
    subprocess.check_call([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-cubin",
                           "-I", os.path.join(ROOT, "helmholtz_preconditioner_b200", "csrc"), "-o", str(cubin), str(src)])
    sass = subprocess.check_output([cuobjdump, "-sass", str(cubin)], text=True)
    instr = [ln.split("*/", 1)[1].split(";")[0].strip() for ln in sass.splitlines() if re.match(r"\s*/\*[0-9a-f]{4}\*/", ln)]
    assert not [i for i in instr if re.match(r"CALL\b", i)], sass
    assert len([i for i in instr if re.match(r"ATOMG\S*\.EXCH\b", i)]) == 2, sass
