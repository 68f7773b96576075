"""CPU: the C-ABI library loads, exports every symbol include/ekpose_b200.h declares, fails loudly
without a GPU, and the product never routes through the oracle."""
import ctypes
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "ekpose_b200.h")
SO = os.path.join(ROOT, "torch_ekpose_b200", "libekpose_b200.so")


def declared_symbols():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    names = re.findall(r"^\s*(?:const\s+)?(?:int|void|float|long long|char)\s*\*?\s*(\w+)\s*\(", src, flags=re.M)
    return sorted(set(names))


def test_header_declares_the_reference_surface():
    names = declared_symbols()
    for n in ("process_paf", "get_num_humans", "get_part_cid", "get_score", "get_part_x", "get_part_y", "get_part_score"):
        assert n in names        # lib/pafprocess/pafprocess.h:53-59
    assert len(names) >= 20


def test_library_exports_every_declared_symbol():
    assert os.path.exists(SO), "build first: make -C torch_ekpose_b200/csrc"
    lib = ctypes.CDLL(SO)
    for n in declared_symbols():
        assert hasattr(lib, n), f"{n} declared in ekpose_b200.h but not exported"
    out = subprocess.run(["nm", "-D", "--defined-only", SO], capture_output=True, text=True).stdout
    exported = {l.split()[-1] for l in out.splitlines() if " T " in l}
    assert set(declared_symbols()) <= exported


def test_python_binding_covers_the_header():
    from torch_ekpose_b200 import _lib
    assert sorted(_lib.SIGNATURES) == declared_symbols()


def test_sass_is_sm_100a_only():
    # next to the nvcc torch_ekpose_b200/csrc/Makefile builds with (NVCC ?= /usr/local/cuda/bin/nvcc), on PATH or not
    nvcc = shutil.which(os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc"))
    assert nvcc, "the nvcc the library was built with is not found"
    cuobjdump = os.path.join(os.path.dirname(nvcc), "cuobjdump")
    out = subprocess.run([cuobjdump, "-lelf", SO], capture_output=True, text=True).stdout
    archs = set(re.findall(r"sm_(\d+a?)", out))
    assert archs == {"100a"}, archs


def _no_gpu():
    try:
        import torch
        return not torch.cuda.is_available()
    except Exception:
        return True


@pytest.mark.skipif(not _no_gpu(), reason="checks the no-GPU behaviour")
def test_no_cpu_fallback_fails_loudly():
    import torch_ekpose_b200 as ek
    with pytest.raises(ek._lib.EkpError) as e:
        ek.pafprocess.process_paf(np.zeros((1, 2, 5), np.float32), np.zeros((8, 8, 19), np.float32), np.zeros((8, 8, 38), np.float32))
    assert e.value.code == ek._lib.ERR_CUDA and "no CPU fallback" in str(e.value)
    with pytest.raises(ek._lib.EkpError):
        ek.PostProcessor(device=0)
    with pytest.raises(ek._lib.EkpError):
        ek.paf_to_pose_cpp(np.zeros((46, 54, 19), np.float32), np.zeros((46, 54, 38), np.float32))
    assert ek.pafprocess.get_num_humans() == 0


def test_argument_conversion_mirrors_numpy_i():
    import torch_ekpose_b200 as ek
    with pytest.raises(TypeError):   # numpy.i require_dimensions: ndim must be 3
        ek.pafprocess.process_paf(np.zeros((2, 5), np.float32), np.zeros((8, 8, 19)), np.zeros((8, 8, 38)))
    with pytest.raises(TypeError):
        ek.pafprocess.process_paf(np.zeros((1, 2, 5)), np.zeros((8, 8, 19)), "not an array")


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "torch_ekpose_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cpp")) or f == "Makefile":
                text = open(os.path.join(dirpath, f), errors="ignore").read()
                assert not re.search(r"^\s*(import|from)\s+oracle", text, flags=re.M), f
                assert "libekp_oracle" not in text and "libpaf_ref" not in text, f
                assert not re.search(r'#include\s+"[^"]*oracle', text), f


def _build_c_example(tmp_path):
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = str(tmp_path / "c_abi_example")
    cmd = ["gcc", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-I", os.path.join(root, "include"),
           os.path.join(root, "tools", "c_abi_example.c"), "-L", os.path.join(root, "torch_ekpose_b200"), "-lekpose_b200",
           "-Wl,-rpath," + os.path.join(root, "torch_ekpose_b200"), "-o", exe]
    out = subprocess.run(cmd, capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    return subprocess.run([exe], capture_output=True, text=True, timeout=120)


def test_header_is_plain_c_and_links(tmp_path):
    """include/ekpose_b200.h compiles as pedantic C99 and a C program links against the library's seven reference
    symbols; without a GPU it reports EKP_ERR_CUDA (exit 3), with one it prints the known answer."""
    run = _build_c_example(tmp_path)
    try:
        import torch
        have_gpu = torch.cuda.is_available()
    except Exception:
        have_gpu = False
    if have_gpu:
        assert run.returncode == 0 and "humans 1, score 1.500" in run.stdout, run.stdout + run.stderr
    else:
        assert run.returncode == 3 and "no CPU fallback" in run.stderr, run.stdout + run.stderr


@pytest.mark.gpu
def test_c_caller_known_answer(tmp_path):
    """The C99 caller of tools/c_abi_example.c on the GPU: SURVEY.md Appendix A.6 (1 human, score 1.5, x of cid 3 = 40)."""
    run = _build_c_example(tmp_path)
    assert run.returncode == 0, run.stdout + run.stderr
    assert "humans 1, score 1.500, parts 1..4 -> cids 0 1 2 3, x of cid 3 = 40" in run.stdout
