"""ctypes binding of libkbp.so (the C ABI in include/kbp.h) -- the only way numerical work leaves
Python in this package.  There is NO CPU fallback: if the library or a CUDA device is missing,
``Engine()`` raises ``EngineUnavailable`` and every compute entry point of the package fails loudly.
"""
from __future__ import annotations

import ctypes
import os
import threading

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("KBP_LIB") or os.path.join(_HERE, "libkbp.so")      # KBP_LIB: developer override (debug builds)

OP_PERMUTE, OP_GEMM, OP_QR, OP_SVD, OP_NORMALIZE, OP_EMBED, OP_ZERO, OP_SCALAR_TO_SLOT, OP_NONFINITE, OP_EYE, OP_SU = range(1, 12)
E_SVD_NOCONV, E_NONFINITE = -4, -5

EXPORTED = [
    "kbp_create", "kbp_destroy", "kbp_last_error", "kbp_device_count", "kbp_reserve", "kbp_upload", "kbp_download",
    "kbp_broadcast", "kbp_slots_read", "kbp_slots_zero", "kbp_run", "kbp_sync", "kbp_svd_work_elems",
    "kbp_qr_work_elems", "kbp_svd_warm_elems", "kbp_launch_count", "kbp_gemm_flops", "kbp_svd_sweeps", "kbp_svd_counters", "kbp_timer_start", "kbp_timer_stop_ms",
    "kbp_profile_enable", "kbp_profile_read", "kbp_graph_ready", "kbp_graph_counters", "kbp_graph_policy", "kbp_ktime_report", "kbp_arena_ptr", "kbp_slots_ptr", "kbp_stream_ptr", "kbp_chain_elems",
]


class EngineUnavailable(RuntimeError):
    pass


class BubbleConError(RuntimeError):
    """raised where the reference prints and calls exit(1) (src/libs/bubblecon.py:2921-2949,
    src/libs/bmpslib.py:711-717); name follows src/_error_types.py."""


def raise_if_not_converged(rc: int, where: str = ""):
    """A truncation built from a factorisation that did not converge must not flow on silently (the reference retries a
    failed SVD with a perturbed matrix and exits if that fails too, src/libs/bmpslib.py:741-745)."""
    if rc == E_SVD_NOCONV:
        raise BubbleConError(f"truncated SVD did not converge on the device{': ' + where if where else ''}")


_lib = None
_lib_lock = threading.Lock()


def load_library():
    global _lib
    with _lib_lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise EngineUnavailable(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc -gencode arch=compute_100a,code=sm_100a).  There is no CPU fallback.")
        lib = ctypes.CDLL(LIB_PATH)
        P, I, L, D = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_double
        lib.kbp_create.argtypes = [I, ctypes.POINTER(P)]; lib.kbp_create.restype = I
        lib.kbp_destroy.argtypes = [P]; lib.kbp_destroy.restype = None
        lib.kbp_last_error.argtypes = [P]; lib.kbp_last_error.restype = ctypes.c_char_p
        lib.kbp_device_count.argtypes = []; lib.kbp_device_count.restype = I
        lib.kbp_reserve.argtypes = [P, L, I, I]; lib.kbp_reserve.restype = I
        lib.kbp_upload.argtypes = [P, I, L, P, L]; lib.kbp_upload.restype = I
        lib.kbp_download.argtypes = [P, I, L, P, L]; lib.kbp_download.restype = I
        lib.kbp_broadcast.argtypes = [P, L, P, L]; lib.kbp_broadcast.restype = I
        lib.kbp_slots_read.argtypes = [P, P]; lib.kbp_slots_read.restype = I
        lib.kbp_slots_zero.argtypes = [P]; lib.kbp_slots_zero.restype = I
        lib.kbp_run.argtypes = [P, P, L]; lib.kbp_run.restype = I
        lib.kbp_graph_ready.argtypes = [P, P, L]; lib.kbp_graph_ready.restype = I
        lib.kbp_graph_counters.argtypes = [P, P]; lib.kbp_graph_counters.restype = I
        lib.kbp_ktime_report.argtypes = [P, ctypes.c_char_p]; lib.kbp_ktime_report.restype = I
        lib.kbp_graph_policy.argtypes = [P, L, I]; lib.kbp_graph_policy.restype = I
        for nm in ("kbp_arena_ptr", "kbp_slots_ptr", "kbp_stream_ptr"):
            getattr(lib, nm).argtypes = [P]; getattr(lib, nm).restype = ctypes.c_uint64
        lib.kbp_chain_elems.argtypes = [P]; lib.kbp_chain_elems.restype = L
        lib.kbp_sync.argtypes = [P]; lib.kbp_sync.restype = I
        lib.kbp_svd_work_elems.argtypes = [L, L]; lib.kbp_svd_work_elems.restype = L
        lib.kbp_qr_work_elems.argtypes = [L, L]; lib.kbp_qr_work_elems.restype = L
        lib.kbp_svd_warm_elems.argtypes = [L, L, L]; lib.kbp_svd_warm_elems.restype = L
        lib.kbp_launch_count.argtypes = [P]; lib.kbp_launch_count.restype = L
        lib.kbp_gemm_flops.argtypes = [P]; lib.kbp_gemm_flops.restype = D
        lib.kbp_svd_sweeps.argtypes = [P]; lib.kbp_svd_sweeps.restype = L
        lib.kbp_svd_counters.argtypes = [P, P]; lib.kbp_svd_counters.restype = I
        lib.kbp_timer_start.argtypes = [P]; lib.kbp_timer_start.restype = I
        lib.kbp_timer_stop_ms.argtypes = [P, ctypes.POINTER(D)]; lib.kbp_timer_stop_ms.restype = I
        lib.kbp_profile_enable.argtypes = [P, I]; lib.kbp_profile_enable.restype = I
        lib.kbp_profile_read.argtypes = [P, P, P]; lib.kbp_profile_read.restype = I
        _lib = lib
        return lib


def svd_work_elems(m: int, n: int) -> int:
    """pure-integer mirror of kbp_svd_work_elems so programs can be compiled without a device."""
    p, q = (n, m) if m >= n else (m, n)
    p_pad = (p + 31) // 32 * 32
    q_pad = (q + 7) // 8 * 8
    jacobi = p_pad * (q_pad + p_pad)
    subspace = 6 * q_pad * 192 + 17 * 192 * 192 + m * n + 64      # k_tsvd.cu: tsvd_work_elems
    return max(jacobi, subspace)


def svd_warm_elems(m: int, n: int, keep: int) -> int:
    """reserved (mirrors kbp_svd_warm_elems): KBP_OP_SVD keeps no state between runs."""
    return 0


def qr_work_elems(m: int, n: int) -> int:
    k = min(m, n)
    return m * n + m * k + k + 8


class _CudaArray:
    def __init__(self, ptr, n, typestr):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": typestr, "data": (ptr, False), "version": 2}


def _cuda_view(ptr: int, n: int, typestr: str, device: int):
    import torch
    with torch.cuda.device(device):
        return torch.as_tensor(_CudaArray(ptr, n, typestr), device=torch.device("cuda", device))


class Engine:
    """one CUDA context-stream + device arena holding ``nb`` chains."""

    def __init__(self, device: int = 0):
        self.lib = load_library()
        if self.lib.kbp_device_count() <= 0:
            raise EngineUnavailable("no CUDA device visible: the block-BP engine has no CPU fallback")
        h = ctypes.c_void_p()
        rc = self.lib.kbp_create(device, ctypes.byref(h))
        if rc != 0:
            raise EngineUnavailable(f"kbp_create(device={device}) failed with code {rc}")
        self.h = h
        self.device = device
        self.nb = 0
        self.n_slots = 0
        self.chain_elems = 0

    def close(self):
        if getattr(self, "h", None):
            self.lib.kbp_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, soft=()):
        if rc == 0 or rc in soft:
            return rc
        raise BubbleConError(f"libkbp error {rc}: {self.lib.kbp_last_error(self.h).decode()}")

    def reserve(self, chain_elems: int, nb: int, n_slots: int = 16):
        self._check(self.lib.kbp_reserve(self.h, int(chain_elems), int(nb), int(n_slots)))
        self.nb, self.n_slots = nb, n_slots
        self.chain_elems = int(chain_elems)

    def upload(self, offset: int, arr: np.ndarray, chain: int = -1):
        """``arr``: [nb, n] (chain=-1) or [n] complex128."""
        a = np.ascontiguousarray(arr, dtype=np.complex128)
        n = a.shape[-1] if chain < 0 else a.size
        if chain < 0:
            assert a.ndim == 2 and a.shape[0] == self.nb
        self._check(self.lib.kbp_upload(self.h, chain, int(offset), a.ctypes.data_as(ctypes.c_void_p), int(n)))

    def broadcast(self, offset: int, arr: np.ndarray):
        a = np.ascontiguousarray(arr, dtype=np.complex128).ravel()
        self._check(self.lib.kbp_broadcast(self.h, int(offset), a.ctypes.data_as(ctypes.c_void_p), int(a.size)))

    def download(self, offset: int, n: int, chain: int = -1) -> np.ndarray:
        out = np.empty((self.nb, n) if chain < 0 else (n,), dtype=np.complex128)
        self._check(self.lib.kbp_download(self.h, chain, int(offset), out.ctypes.data_as(ctypes.c_void_p), int(n)))
        return out

    def slots(self) -> np.ndarray:
        out = np.empty((self.nb, self.n_slots), dtype=np.float64)
        self._check(self.lib.kbp_slots_read(self.h, out.ctypes.data_as(ctypes.c_void_p)))
        return out

    def slots_zero(self):
        self._check(self.lib.kbp_slots_zero(self.h))

    def run(self, words: np.ndarray, soft_errors=()):
        w = np.ascontiguousarray(words, dtype=np.int64)
        return self._check(self.lib.kbp_run(self.h, w.ctypes.data_as(ctypes.c_void_p), int(w.size)), soft=soft_errors)

    def ktime_report(self, tag: str = ""):
        self.lib.kbp_ktime_report(self.h, tag.encode())

    def spec_counters(self) -> dict:
        """zero counts, without calling the library: bench.py calls it and reports these keys in its ``svd_paths`` block."""
        return {"spec_launches": 0, "spec_failures": 0}

    def graph_ready(self, words: np.ndarray) -> bool:
        """True: the next ``run`` of this program is one asynchronous CUDA-graph launch (no host decisions)."""
        w = np.ascontiguousarray(words, dtype=np.int64)
        return bool(self.lib.kbp_graph_ready(self.h, w.ctypes.data_as(ctypes.c_void_p), int(w.size)))

    # ---- zero-copy views for the multi-GPU message exchange (torch is plumbing here: device memory + NCCL) ----
    def arena_tensor(self):
        """the arena as a flat torch complex128 CUDA tensor [nb * chain_elems] sharing the engine's memory."""
        return _cuda_view(int(self.lib.kbp_arena_ptr(self.h)), self.nb * int(self.lib.kbp_chain_elems(self.h)), "<c16", self.device)

    def slots_tensor(self):
        return _cuda_view(int(self.lib.kbp_slots_ptr(self.h)), self.nb * self.n_slots, "<f8", self.device)

    def torch_stream(self):
        import torch
        return torch.cuda.ExternalStream(int(self.lib.kbp_stream_ptr(self.h)), device=torch.device("cuda", self.device))

    def graph_policy(self, min_words: int = 256, capture_first: bool = False):
        self._check(self.lib.kbp_graph_policy(self.h, int(min_words), 1 if capture_first else 0))

    def graph_counters(self) -> dict:
        out = np.zeros(4, dtype=np.int64)
        self._check(self.lib.kbp_graph_counters(self.h, out.ctypes.data_as(ctypes.c_void_p)))
        return {"graph_replays": int(out[0]), "graph_captures": int(out[1]), "graphs_alive": int(out[2]), "graph_capture_failures": int(out[3])}

    def sync(self):
        self._check(self.lib.kbp_sync(self.h))

    def launch_count(self) -> int:
        return int(self.lib.kbp_launch_count(self.h))

    def gemm_flops(self) -> float:
        """real flops executed so far by the ZGEMM launches of this engine (include/kbp.h: kbp_gemm_flops)."""
        return float(self.lib.kbp_gemm_flops(self.h))

    def svd_sweeps(self) -> int:
        return int(self.lib.kbp_svd_sweeps(self.h))

    def svd_counters(self) -> dict:
        """how the truncations were executed so far (synchronises): in-smem Jacobi / Householder-reduced / subspace iteration /
        its hand-overs to the exact path / block-Jacobi runs; the device-decided ones are counted by the decision kernels."""
        out = np.zeros(8, dtype=np.int64)
        self._check(self.lib.kbp_svd_counters(self.h, out.ctypes.data_as(ctypes.c_void_p)))
        d = {"small": int(out[1]), "reduced": int(out[0]), "subspace": int(out[2]), "subspace_fallback": int(out[3]),
             "block_jacobi": int(out[4]), "subspace_iterations": int(out[5]), "block_jacobi_sweeps": int(out[6]),
             "not_converged": int(out[7])}
        d.update(self.graph_counters())
        return d

    def profile_enable(self, on: bool):
        self._check(self.lib.kbp_profile_enable(self.h, 1 if on else 0))

    def profile_read(self):
        ms = np.zeros(16)
        cnt = np.zeros(16, dtype=np.int64)
        self._check(self.lib.kbp_profile_read(self.h, ms.ctypes.data_as(ctypes.c_void_p), cnt.ctypes.data_as(ctypes.c_void_p)))
        return ms, cnt

    def timer_start(self):
        self._check(self.lib.kbp_timer_start(self.h))

    def timer_stop_ms(self) -> float:
        ms = ctypes.c_double()
        self._check(self.lib.kbp_timer_stop_ms(self.h, ctypes.byref(ms)))
        return float(ms.value)
