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


def test_evaluation_launches_take_their_stream_and_job_table_from_their_arguments():
    """The evaluation launchers read the stream they issue on, the pose table and its host mirrors from their JobSet
    argument: the context holds no view that a caller repoints while a call runs, and every launch is counted once,
    where it is issued."""
    import glob
    import re
    ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    csrc = os.path.join(ROOT, "nid-pose-estimation_b200", "csrc")

    def code(path):
        src = re.sub(r'"(?:\\.|[^"\\])*"', '""', open(path).read())
        return re.sub(r"//[^\n]*|/\*.*?\*/", "", src, flags=re.S)

    sources = {os.path.basename(p): code(p) for p in sorted(glob.glob(os.path.join(csrc, "*.cu*")) + glob.glob(os.path.join(csrc, "*.h")))}
    hdr = sources["nid_ctx.h"]
    ctx = re.search(r"struct nid_ctx \{(.*?)\n\};", hdr, re.S).group(1)
    views = re.findall(r"\b(poses|h_poses|h_job_pair)\s*[=;\[]", ctx)
    assert not views, views
    # a context's stream is created once and never assigned: find every name a nid_ctx pointer goes by
    names = set()
    for src in sources.values():
        names |= set(re.findall(r"\bnid_ctx\s*\*\s*(?:const\s*\*?\s*)?(\w+)", src))
    assert {"c", "dst", "src"} <= names
    assigned = [(f, m) for f, src in sources.items()
                for m in re.findall(r"\b(?:%s)->stream\s*=(?!=)" % "|".join(sorted(names)), src)]
    assert not assigned, assigned
    decrements = [f for f, src in sources.items() if re.search(r"launches\s*(--|-=)", src)]
    assert not decrements, decrements
    launchers = {"launch_pass1", "launch_pass2", "launch_gn", "launch_sorted_tail_gn", "launch_latency_round", "launch_hard",
                 "launch_warp_sample_jobs"}
    decl = dict(re.findall(r"\bint (launch_\w+)\(([^)]*)\);", hdr))
    assert launchers <= set(decl), launchers - set(decl)
    wrong = [n for n in sorted(launchers) if "const JobSet&" not in decl[n]]
    assert not wrong, wrong


def test_the_huber_threshold_is_rounded_in_one_place():
    """The reference keeps delta^2 as a float (robust_kernel_impl.h:84). The device code rounds it in one helper,
    huber_dsqr in nid_ctx.h, and every launcher of a Gauss-Newton kernel fills EvalParams::huber_dsqr from it: the
    blocks of k_gn, k_tail_gn and k_gn_out classify a cell by the same value, the one
    tests/test_gpu_large_grids_gn.py::test_float_dsqr_on_the_device pins."""
    import glob
    import re
    ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    csrc = os.path.join(ROOT, "nid-pose-estimation_b200", "csrc")
    sources = {}
    for path in sorted(glob.glob(os.path.join(csrc, "*.cu*")) + glob.glob(os.path.join(csrc, "*.h"))):
        src = re.sub(r'"(?:\\.|[^"\\])*"', '""', open(path).read())
        sources[os.path.basename(path)] = re.sub(r"//[^\n]*|/\*.*?\*/", "", src, flags=re.S)
    casts = [(f, m) for f, src in sources.items() for m in re.findall(r"\(float\)\s*\(\s*delta\b[^;]*", src)]
    assert casts == [("nid_ctx.h", "(float)(delta * delta)")], casts
    assert re.search(r"inline double huber_dsqr\(double delta\) \{ return \(double\)\(float\)\(delta \* delta\); \}",
                     sources["nid_ctx.h"])
    fills = [(f, m.strip()) for f, src in sorted(sources.items()) for m in re.findall(r"\.huber_dsqr\s*=([^;]*);", src)]
    assert fills == [("nid_kernels.cu", "huber_dsqr(delta)"), ("nid_sorted.cu", "huber_dsqr(delta)")], fills
