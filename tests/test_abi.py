"""CPU-side checks of the drop-in boundary: the shared library loads, exports every symbol that
include/nid_b200.h declares plus the three reference-signature C++ entry points, and fails loudly
(instead of falling back to a CPU path) when there is no CUDA device."""
import ctypes
import os
import subprocess

import pytest


def test_library_exports_every_declared_symbol(nid):
    L = nid.lib()
    names = nid.exported_symbols_in_header()
    assert len(names) >= 25
    missing = [n for n in names if not hasattr(L, n)]
    assert not missing, missing


def test_reference_signature_shims_are_exported(nid):
    out = subprocess.check_output(["nm", "-D", "--defined-only", nid.LIB_PATH]).decode()
    # Calculate3Dpoint(double*,double*,double*,double*,int,int)            CudaPoints3d.cuh:6
    assert "_Z16Calculate3DpointPdS_S_S_ii" in out
    # CudaComputeHref(double*,double*,double*,double*,int x5,double*,int*,int*,double*)  CudaComputeHref.cuh:6
    assert "_Z15CudaComputeHrefPdS_S_S_iiiiiS_PiS0_S_" in out
    # g2o::CudaComputeH(bool,double* x3,int*,double*,int*,double*,double*,int x5,double* x6)  computeH.cuh:8
    assert "_ZN3g2o12CudaComputeHEbPdS0_S0_PiS0_S1_S0_S0_iiiiiS0_S0_S0_S0_S0_S0_" in out


def test_product_does_not_link_the_oracle(nid):
    out = subprocess.check_output(["nm", "-D", nid.LIB_PATH]).decode()
    assert "orc_" not in out
    ldd = subprocess.check_output(["ldd", nid.LIB_PATH]).decode()
    assert "oracle" not in ldd


def test_bad_arguments_are_rejected_without_touching_the_gpu(nid):
    L = nid.lib()
    h = ctypes.c_void_p()
    assert L.nid_create(ctypes.byref(h), 0, 480, 640, 4, 16, 2, 1, 1) == -4  # degree != 3
    assert b"degree" in L.nid_last_error()
    assert L.nid_create(ctypes.byref(h), 0, 480, 640, 0, 16, 3, 1, 1) == -2
    assert L.nid_create(ctypes.byref(h), 0, 480, 640, 4, 3, 3, 1, 1) == -2


def test_no_cpu_fallback(nid):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(nid.NidError, match="no CUDA device"):
        nid.Context(120, 160, 4, 16)


def test_every_run_time_option_is_documented_in_the_header():
    """nid_set_option's keys are part of the interface: every key the library accepts is described in include/nid_b200.h."""
    import re
    ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = open(os.path.join(ROOT, "nid-pose-estimation_b200", "csrc", "nid_api.cu")).read()
    keys = set(re.findall(r'strcmp\(key, "([a-z_0-9]+)"\)', src))
    assert {"path", "task_px", "lm_speculate", "lm_graph"} <= keys
    hdr = open(os.path.join(ROOT, "include", "nid_b200.h")).read()
    missing = [k for k in sorted(keys) if f'"{k}"' not in hdr]
    assert not missing, missing


def test_cuda_resources_are_acquired_and_released_only_by_their_owner_types():
    """A context's device and pinned buffers, streams, events, arrays, textures and graphs are held by the owner types of
    csrc/nid_handles.h, which release them in their destructors: no source file allocates or releases one by hand, so a
    context frees everything it holds on every way out, a nid_create that fails half way included."""
    import glob
    import re
    ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    csrc = os.path.join(ROOT, "nid-pose-estimation_b200", "csrc")
    release = {"cudaFree", "cudaFreeHost", "cudaFreeArray", "cudaEventDestroy", "cudaStreamDestroy",
               "cudaDestroyTextureObject", "cudaGraphDestroy", "cudaGraphExecDestroy"}
    acquire = {"cudaMalloc", "cudaMallocHost", "cudaMallocArray", "cudaCreateTextureObject", "cudaStreamCreate",
               "cudaStreamCreateWithFlags", "cudaEventCreate", "cudaEventCreateWithFlags"}
    found = {}
    for path in sorted(glob.glob(os.path.join(csrc, "*.cu*")) + glob.glob(os.path.join(csrc, "*.h"))):
        code = re.sub(r'"(?:\\.|[^"\\])*"', '""', open(path).read())  # (error texts name the calls they report)
        code = re.sub(r"//[^\n]*|/\*.*?\*/", "", code, flags=re.S)
        names = set(re.findall(r"\bcuda\w+", code)) & (release | acquire)
        if names:
            found[os.path.basename(path)] = names
    assert set(found) == {"nid_handles.h"}, found
    assert release <= found["nid_handles.h"]
