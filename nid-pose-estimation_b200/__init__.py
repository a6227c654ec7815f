"""nid-pose-estimation_b200 — B200-native NID cost + Jacobian path.

Thin ctypes mirror of include/nid_b200.h (the C-ABI of csrc/, built by `make` in this directory into
libnid_b200.so). There is no Python or CPU implementation behind it: if the CUDA library is missing or
no GPU is present the calls raise.

The directory name is not a Python identifier; import it with
    importlib.import_module("nid-pose-estimation_b200")
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("NID_B200_LIB") or os.path.join(_HERE, "libnid_b200.so")
HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "nid_b200.h")

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int)
_u8p = C.POINTER(C.c_uint8)
_fp = C.POINTER(C.c_float)

_lib = None


class NidError(RuntimeError):
    pass


def build(verbose: bool = False) -> str:
    """Compile the CUDA library for sm_100a (nvcc cross-compiles without a GPU)."""
    subprocess.check_call(["make", "-C", _HERE, "libnid_b200.so"], stdout=None if verbose else subprocess.DEVNULL)
    return LIB_PATH


def lib():
    """Load libnid_b200.so. Raises if it has not been built: there is no fallback."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise NidError(f"{LIB_PATH} is missing: build it with `make -C {_HERE}` "
                           "(the NID path has no CPU/PyTorch fallback)")
        L = C.CDLL(LIB_PATH)
        L.nid_last_error.restype = C.c_char_p
        L.nid_create.argtypes = [C.POINTER(C.c_void_p)] + [C.c_int] * 8
        L.nid_destroy.argtypes = [C.c_void_p]
        L.nid_sync.argtypes = [C.c_void_p]
        L.nid_set_pair.argtypes = [C.c_void_p, C.c_int, _dp, _u8p, _u8p, _dp, _dp]
        L.nid_set_pairs_u16.argtypes = [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_uint16), _u8p, _u8p, _dp, _dp]
        L.nid_prepare_pairs.argtypes = [C.c_void_p, C.c_int, C.c_int, _dp, _ip, _dp]
        L.nid_set_target.argtypes = [C.c_void_p, C.c_int, _u8p]
        L.nid_set_pair_f64.argtypes = [C.c_void_p, C.c_int, _dp, _dp, _dp, _dp, _dp]
        L.nid_set_pair_points.argtypes = [C.c_void_p, C.c_int, _dp, _dp, _dp, _dp]
        L.nid_import_prepare.argtypes = [C.c_void_p, C.c_int, _dp, _ip, _dp]
        L.nid_get_inbounds.argtypes = [C.c_void_p, C.c_int, _u8p]
        L.nid_get_points3d.argtypes = [C.c_void_p, C.c_int, _dp]
        L.nid_prepare.argtypes = [C.c_void_p, C.c_int, _dp, _ip, _dp]
        L.nid_get_ref_weights.argtypes = [C.c_void_p, C.c_int, _dp, _ip]
        L.nid_eval.argtypes = [C.c_void_p, C.c_int, _dp, C.c_int, _dp, _dp, _dp]
        L.nid_eval_jobs.argtypes = [C.c_void_p, C.c_int, _ip, _dp, C.c_int, _dp, _dp, _dp]
        L.nid_stage_jobs.argtypes = [C.c_void_p, C.c_int, _ip, _dp]
        L.nid_eval_staged.argtypes = [C.c_void_p, C.c_int, C.c_int]
        L.nid_fetch_results.argtypes = [C.c_void_p, C.c_int, C.c_int, _dp, _dp, _dp]
        L.nid_eval_gn.argtypes = [C.c_void_p, C.c_int, _dp, C.c_double, _dp, _dp, _dp, _dp, _dp]
        L.nid_solve.argtypes = [C.c_void_p, C.c_int, _dp, C.c_int, C.c_double, _dp, _ip]
        L.nid_solve_jobs.argtypes = [C.c_void_p, C.c_int, _ip, _dp, C.c_int, C.c_double, _ip]
        L.nid_solve_groups.argtypes = [C.c_void_p, C.c_int, _ip, _ip, _dp, _dp, C.c_int, C.c_double, _ip, _dp]
        L.nid_set_pairs_downsampled.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int]
        L.nid_solve_pyramid_jobs.argtypes = [C.POINTER(C.c_void_p), C.c_int, C.c_int, _ip, _dp, _ip, C.c_double, _ip]
        L.nid_hard_eval_jobs.argtypes = [C.c_void_p, C.c_int, _ip, _dp, _dp, _dp]
        L.nid_warp_sample.argtypes = [C.c_void_p, C.c_int, _dp, _fp]
        L.nid_warp_sample_f64.argtypes = [C.c_void_p, C.c_int, _dp, _dp]
        L.nid_warp_sample_jobs.argtypes = [C.c_void_p, C.c_int, _ip, _dp, _fp]
        L.nid_debug_hist.argtypes = [C.c_void_p, C.c_int, C.c_int, _dp, _dp]
        L.nid_launch_count.restype = C.c_longlong
        L.nid_launch_count.argtypes = [C.c_void_p]
        L.nid_live_resources.restype = C.c_longlong
        L.nid_live_resources.argtypes = []
        L.nid_set_option.argtypes = [C.c_void_p, C.c_char_p, C.c_int]
        L.nid_kernel_times.argtypes = [C.c_void_p, _dp, C.POINTER(C.c_longlong)]
        L.nid_stream.restype = C.c_void_p
        L.nid_stream.argtypes = [C.c_void_p]
        L.nid_event_record.argtypes = [C.c_void_p, C.c_int]
        L.nid_event_elapsed_ms.argtypes = [C.c_void_p, _fp]
        # reference-signature shims, C-linkage trampolines
        L.nid_shim_Calculate3Dpoint.argtypes = [_dp, _dp, _dp, _dp, C.c_int, C.c_int]
        L.nid_shim_CudaComputeHref.argtypes = [_dp, _dp, _dp, _dp] + [C.c_int] * 5 + [_dp, _ip, _ip, _dp]
        L.nid_shim_CudaComputeH.argtypes = ([C.c_int, _dp, _dp, _dp, _ip, _dp, _ip, _dp, _dp] + [C.c_int] * 5 +
                                            [_dp] * 6)
        _lib = L
    return _lib


def _chk(rc: int):
    if rc != 0:
        raise NidError(f"nid_b200 error {rc}: {lib().nid_last_error().decode()}")


def _d(a):
    return a.ctypes.data_as(_dp)


def _f64(a, n=None):
    a = np.ascontiguousarray(a, dtype=np.float64)
    if n is not None and a.size != n:
        raise ValueError(f"expected {n} doubles, got {a.size}")
    return a


class Context:
    """One `nid_ctx`: `n_pairs` frame pairs of one geometry, up to `max_jobs` evaluations per submission."""

    def __init__(self, rows, cols, cell, bins, n_pairs=1, max_jobs=1, device=0, degree=3):
        self.rows, self.cols, self.cell, self.bins = rows, cols, cell, bins
        self.ncell = cell * cell
        self.n = rows * cols
        self.n_pairs, self.max_jobs = n_pairs, max_jobs
        h = C.c_void_p()
        _chk(lib().nid_create(C.byref(h), device, rows, cols, cell, bins, degree, n_pairs, max_jobs))
        self._h = h

    def close(self):
        if getattr(self, "_h", None):
            lib().nid_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- a1
    def set_pair(self, pair, depth, im0, im1, T_wc0, intr):
        im0 = np.ascontiguousarray(im0, dtype=np.uint8)
        im1 = np.ascontiguousarray(im1, dtype=np.uint8)
        _chk(lib().nid_set_pair(self._h, pair, _d(_f64(depth, self.n)), im0.ctypes.data_as(_u8p),
                                im1.ctypes.data_as(_u8p), _d(_f64(T_wc0, 16)), _d(_f64(intr, 5))))

    def set_pairs_u16(self, pair0, depth_raw, im0, im1, T_wc0, intr):
        """Batched, asynchronous set-up of pairs [pair0, pair0 + n) from raw 16-bit depth and 8-bit images
        ([n, rows, cols] each; T_wc0 [n, 16]; intr [n, 5]). The arrays must stay alive and untouched until sync() or
        prepare_pairs(); they are returned so that the caller can hold on to them."""
        d = np.ascontiguousarray(depth_raw, dtype=np.uint16)
        a = np.ascontiguousarray(im0, dtype=np.uint8)
        b = np.ascontiguousarray(im1, dtype=np.uint8)
        n = d.size // self.n
        if d.size != n * self.n or a.size != d.size or b.size != d.size:
            raise ValueError("depth_raw, im0, im1 must hold n * rows * cols elements each")
        T = _f64(T_wc0, 16 * n)
        K = _f64(intr, 5 * n)
        _chk(lib().nid_set_pairs_u16(self._h, pair0, n, d.ctypes.data_as(C.POINTER(C.c_uint16)), a.ctypes.data_as(_u8p),
                                     b.ctypes.data_as(_u8p), _d(T), _d(K)))
        return d, a, b, T, K

    def prepare_pairs(self, pair0, T_cw1):
        """a2 of pairs [pair0, pair0 + n) in one submission -> (n_c [n, cell^2], H_ref [n, cell^2])."""
        T = _f64(T_cw1)
        n = T.size // 16
        nc = np.zeros((n, self.ncell), dtype=np.int32)
        href = np.zeros((n, self.ncell))
        _chk(lib().nid_prepare_pairs(self._h, pair0, n, _d(T), nc.ctypes.data_as(_ip), _d(href)))
        return nc, href

    def set_pairs_downsampled(self, pair0, src, src_pair0, n=1):
        """Fill pairs [pair0, pair0 + n) with the 2x2-downsampled pairs [src_pair0, src_pair0 + n) of Context `src`
        (device to device, asynchronous; prepare before use)."""
        _chk(lib().nid_set_pairs_downsampled(self._h, pair0, src._h if src is not None else None, src_pair0, n))

    def set_target(self, pair, im1):
        """Replace only the target image of a pair (reference-frame reuse); prepare() must be called again."""
        im1 = np.ascontiguousarray(im1, dtype=np.uint8)
        if im1.size != self.n:
            raise ValueError(f"expected {self.n} pixels, got {im1.size}")
        _chk(lib().nid_set_target(self._h, pair, im1.ctypes.data_as(_u8p)))

    def set_pair_f64(self, pair, depth, im0, im1, T_wc0, intr):
        _chk(lib().nid_set_pair_f64(self._h, pair, _d(_f64(depth, self.n)), _d(_f64(im0, self.n)),
                                    _d(_f64(im1, self.n)), _d(_f64(T_wc0, 16)), _d(_f64(intr, 5))))

    def points3d(self, pair=0):
        out = np.zeros(3 * self.n)
        _chk(lib().nid_get_points3d(self._h, pair, _d(out)))
        return out

    # ---- a2
    def prepare(self, pair, T_cw1):
        nc = np.zeros(self.ncell, dtype=np.int32)
        href = np.zeros(self.ncell)
        _chk(lib().nid_prepare(self._h, pair, _d(_f64(T_cw1, 16)), nc.ctypes.data_as(_ip), _d(href)))
        return nc, href

    def ref_weights(self, pair=0):
        bv = np.zeros(4 * self.n)
        bi = np.zeros(self.n, dtype=np.int32)
        _chk(lib().nid_get_ref_weights(self._h, pair, _d(bv), bi.ctypes.data_as(_ip)))
        return bv, bi

    # ---- a9
    def eval(self, pair, T_cw1, want_jac=True):
        Ht, Hj = np.zeros(self.ncell), np.zeros(self.ncell)
        der = np.full(6 * self.ncell, np.nan)
        _chk(lib().nid_eval(self._h, pair, _d(_f64(T_cw1, 16)), int(want_jac), _d(Ht), _d(Hj), _d(der)))
        return Ht, Hj, der.reshape(self.ncell, 6)

    def eval_jobs(self, poses, job_pair=None, want_jac=True):
        poses = _f64(poses)
        n = poses.size // 16
        jp = None if job_pair is None else np.ascontiguousarray(job_pair, dtype=np.int32)
        # (the library writes every element of Ht, Hj and, with want_jac, of der: no need to clear them first)
        Ht, Hj = np.empty((n, self.ncell)), np.empty((n, self.ncell))
        der = np.empty((n, self.ncell, 6)) if want_jac else np.full((n, self.ncell, 6), np.nan)
        _chk(lib().nid_eval_jobs(self._h, n, None if jp is None else jp.ctypes.data_as(_ip), _d(poses), int(want_jac),
                                 _d(Ht), _d(Hj), _d(der)))
        return Ht, Hj, der

    def stage_jobs(self, poses, job_pair=None):
        poses = _f64(poses)
        n = poses.size // 16
        jp = None if job_pair is None else np.ascontiguousarray(job_pair, dtype=np.int32)
        _chk(lib().nid_stage_jobs(self._h, n, None if jp is None else jp.ctypes.data_as(_ip), _d(poses)))
        return n

    def eval_staged(self, n_jobs, want_jac=True):
        _chk(lib().nid_eval_staged(self._h, n_jobs, int(want_jac)))

    def fetch_results(self, n_jobs, want_jac=True):
        Ht, Hj = np.zeros((n_jobs, self.ncell)), np.zeros((n_jobs, self.ncell))
        der = np.full((n_jobs, self.ncell, 6), np.nan)
        _chk(lib().nid_fetch_results(self._h, n_jobs, int(want_jac), _d(Ht), _d(Hj), _d(der)))
        return Ht, Hj, der

    def sync(self):
        _chk(lib().nid_sync(self._h))

    def stream(self) -> int:
        return int(lib().nid_stream(self._h) or 0)

    # ---- a10/a11
    def eval_gn(self, pair, T_cw1, delta):
        chi2 = C.c_double(0)
        H, b = np.zeros(36), np.zeros(6)
        err, J = np.zeros(self.ncell), np.zeros(6 * self.ncell)
        _chk(lib().nid_eval_gn(self._h, pair, _d(_f64(T_cw1, 16)), float(delta), C.byref(chi2), _d(H), _d(b), _d(err),
                               _d(J)))
        return chi2.value, H.reshape(6, 6), b, err, J.reshape(self.ncell, 6)

    def solve(self, pair, pose7, max_iters=10, delta=np.sqrt(0.95)):
        pose = _f64(pose7, 7).copy()
        trace = np.zeros(10 * max_iters)
        stats = np.zeros(3, dtype=np.int32)
        _chk(lib().nid_solve(self._h, pair, _d(pose), max_iters, float(delta), _d(trace), stats.ctypes.data_as(_ip)))
        return pose, trace.reshape(max_iters, 10)[:stats[0]], stats

    def solve_jobs(self, poses7, job_pair=None, max_iters=10, delta=np.sqrt(0.95)):
        poses = _f64(poses7).copy().reshape(-1, 7)
        n = poses.shape[0]
        jp = None if job_pair is None else np.ascontiguousarray(job_pair, dtype=np.int32)
        stats = np.zeros((n, 3), dtype=np.int32)
        _chk(lib().nid_solve_jobs(self._h, n, None if jp is None else jp.ctypes.data_as(_ip), _d(poses), max_iters,
                                  float(delta), stats.ctypes.data_as(_ip)))
        return poses, stats

    def solve_groups(self, poses7, group_sizes, job_pair=None, T_cb=None, max_iters=10, delta=np.sqrt(0.95)):
        """Joint solves (nid_solve_groups): group g's group_sizes[g] jobs share the pose poses7[g] (T_bw); job i is
        evaluated at T_cb[i] @ T_bw (T_cb [n_jobs, 16] column-major, None: identity). Returns (poses [n, 7], stats [n, 3],
        trace [n, max_iters, 10]); the trace rows past stats[g, 0] are zero."""
        poses = _f64(poses7).copy().reshape(-1, 7)
        n = poses.shape[0]
        gs = np.ascontiguousarray(group_sizes, dtype=np.int32).reshape(-1)
        jp = None if job_pair is None else np.ascontiguousarray(job_pair, dtype=np.int32)
        E = None if T_cb is None else _f64(T_cb)
        if gs.size != n:
            raise ValueError(f"{n} poses but {gs.size} group sizes")
        if jp is not None and jp.size != int(gs.sum()):
            raise ValueError(f"{int(gs.sum())} jobs but {jp.size} job pairs")
        if E is not None and E.size != 16 * int(gs.sum()):
            raise ValueError(f"{int(gs.sum())} jobs but {E.size} doubles of T_cb")
        stats = np.zeros((n, 3), dtype=np.int32)
        trace = np.zeros((n, max(max_iters, 0), 10))
        _chk(lib().nid_solve_groups(self._h, n, gs.ctypes.data_as(_ip), None if jp is None else jp.ctypes.data_as(_ip),
                                    None if E is None else _d(E), _d(poses), max_iters, float(delta),
                                    stats.ctypes.data_as(_ip), _d(trace)))
        return poses, stats, trace

    # ---- a12
    def hard_eval_jobs(self, poses, job_pair=None):
        poses = _f64(poses)
        n = poses.size // 16
        jp = None if job_pair is None else np.ascontiguousarray(job_pair, dtype=np.int32)
        total = np.zeros(n)
        cells = np.zeros((n, self.ncell))
        _chk(lib().nid_hard_eval_jobs(self._h, n, None if jp is None else jp.ctypes.data_as(_ip), _d(poses), _d(total),
                                      _d(cells)))
        return total, cells

    # ---- kernel 1
    def warp_sample(self, pair, T_cw1, fetch=True):
        out = np.zeros((self.n, 4), dtype=np.float32) if fetch else None
        _chk(lib().nid_warp_sample(self._h, pair, _d(_f64(T_cw1, 16)), out.ctypes.data_as(_fp) if fetch else None))
        return out

    def warp_sample_jobs(self, poses, job_pair, fetch=True):
        """Kernel-1 record {I_c, g_x, g_y, valid} of every (pair, pose) job in one launch -> [n_jobs, N, 4] float32."""
        poses = _f64(poses).reshape(-1, 16)
        n = poses.shape[0]
        jp = np.ascontiguousarray(job_pair, dtype=np.int32)
        out = np.empty((n, self.rows * self.cols, 4), dtype=np.float32) if fetch else None
        _chk(lib().nid_warp_sample_jobs(self._h, n, jp.ctypes.data_as(_ip), _d(poses),
                                        out.ctypes.data_as(_fp) if fetch else None))
        return out

    def warp_sample_f64(self, pair, T_cw1):
        out = np.zeros((self.n, 8))
        _chk(lib().nid_warp_sample_f64(self._h, pair, _d(_f64(T_cw1, 16)), _d(out)))
        return out

    def debug_hist(self, job, cell_index):
        pt = np.zeros(self.bins)
        pj = np.zeros(self.bins * self.bins)
        _chk(lib().nid_debug_hist(self._h, job, cell_index, _d(pt), _d(pj)))
        return pt, pj.reshape(self.bins, self.bins)

    def event_record(self, slot: int):
        _chk(lib().nid_event_record(self._h, slot))

    def event_elapsed_ms(self) -> float:
        ms = C.c_float(0)
        _chk(lib().nid_event_elapsed_ms(self._h, C.byref(ms)))
        return float(ms.value)

    def kernel_times(self):
        ms = np.zeros(4)
        calls = np.zeros(4, dtype=np.int64)
        _chk(lib().nid_kernel_times(self._h, _d(ms), calls.ctypes.data_as(C.POINTER(C.c_longlong))))
        return dict(zip(("k_hist_sell", "k_jac_sell", "k_jac_final_sorted", "k_assemble"), zip(ms.tolist(), calls.tolist())))

    def launch_count(self) -> int:
        return int(lib().nid_launch_count(self._h))

    def set_option(self, key: str, value: int):
        _chk(lib().nid_set_option(self._h, key.encode(), int(value)))


def solve_pyramid_jobs(levels, poses7, job_pair=None, max_iters=None, delta=np.sqrt(0.95)):
    """Coarse-to-fine solve over Contexts `levels` (finest first): nid_solve_pyramid_jobs. max_iters: one count per level
    (default 10 each). Returns (poses [n, 7], stats [n, n_levels, 3])."""
    L = len(levels)
    poses = _f64(poses7).copy().reshape(-1, 7)
    n = poses.shape[0]
    hs = (C.c_void_p * L)(*[None if c is None else c._h.value for c in levels])
    its = np.ascontiguousarray([10] * L if max_iters is None else max_iters, dtype=np.int32)
    jp = None if job_pair is None else np.ascontiguousarray(job_pair, dtype=np.int32)
    stats = np.zeros((n, L, 3), dtype=np.int32)
    _chk(lib().nid_solve_pyramid_jobs(hs, L, n, None if jp is None else jp.ctypes.data_as(_ip), _d(poses),
                                      its.ctypes.data_as(_ip), float(delta), stats.ctypes.data_as(_ip)))
    return poses, stats


def live_resources() -> int:
    """CUDA resources held by all contexts of the process (nid_live_resources)."""
    return int(lib().nid_live_resources())


def exported_symbols_in_header():
    """Names of every function include/nid_b200.h declares (used by the CPU-side ABI test)."""
    import re
    txt = open(HEADER_PATH).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(nid_[a-z0-9_]+)\s*\(", txt)))
