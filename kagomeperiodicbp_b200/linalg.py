"""Dense linear algebra of the ITE step as device programs: the backend object ``B`` that ``ite.py`` / ``edge_env.py``
are written against.  Every call compiles (once per shape signature) and runs a small tensor program through the C ABI
(include/kbp.h): DMMA ZGEMM for tensordot / scaling / linear combinations, Householder QR, Jacobi SVD, and the Hermitian
eigensolver built on the Jacobi SVD of the shifted matrix.  Arrays cross the boundary as host numpy complex128 (the S3/S4
seams of the reference are per-call host interfaces, SURVEY 8b); reshape / transpose / slicing are host data movement.

There is no CPU fallback: constructing ``DeviceBackend`` without libkbp.so or without a GPU raises ``EngineUnavailable``.
"""
from __future__ import annotations

import math
import os

import numpy as np

from .engine import E_SVD_NOCONV, BubbleConError, raise_if_not_converged
from .program import Program, _prod
from .runtime import Compiled, get_engine

_EIG_SHIFT = 1.5


class DeviceBackend:
    def __init__(self, engine_key="ite-percall", device: int = 0):
        # its own engine: Compiled.load re-reserves the arena and uploads at offset 0, which would overwrite tensors a
        # ResidentBackend on the same engine still holds
        self.eng = get_engine(engine_key, device)
        self._cache: dict = {}
        self.calls = 0

    # ---------------------------------------------------------------- plumbing
    def _run(self, key, build, inputs):
        """build(p, [DT...]) -> list of output DTs; returns list of ndarrays (+ slots)."""
        comp = self._cache.get(key)
        if comp is None:
            p = Program(8)
            dts = [(f"i{k}", p.input(f"i{k}", a.shape if a.ndim else (1,))) for k, a in enumerate(inputs)]
            outs = build(p, [t for _, t in dts])
            comp = Compiled(p, dts, [(f"o{k}", t) for k, t in enumerate(outs)])
            self._cache[key] = comp
        o, sl, rc = comp.run(self.eng, [{f"i{k}": a for k, a in enumerate(inputs)}], soft_errors=(E_SVD_NOCONV,))
        raise_if_not_converged(rc, f"device op {key[0] if isinstance(key, tuple) else key}")
        self.calls += 1
        return [o[0][f"o{k}"] for k in range(len(comp.out_layout))], sl[0]

    @staticmethod
    def _c(a):
        return np.ascontiguousarray(a, dtype=np.complex128)

    # ---------------------------------------------------------------- data movement (host)
    def reshape(self, a, shape):
        return np.reshape(np.asarray(a), shape)

    def transpose(self, a, perm):
        return np.transpose(np.asarray(a), perm)

    # ---------------------------------------------------------------- device ops
    def tensordot(self, a, b, axes, conj_a=False, conj_b=False):
        a, b = self._c(a), self._c(b)
        if isinstance(axes, int):
            assert axes == 0
            out = self.tensordot(a.reshape(-1, 1), b.reshape(1, -1), ([1], [0]), conj_a, conj_b)
            return out.reshape(a.shape + b.shape)
        ax = (tuple(int(x) for x in axes[0]), tuple(int(x) for x in axes[1]))
        if a.size == 0 or b.size == 0:
            return np.tensordot(a, b, axes=ax)
        key = ("td", a.shape, b.shape, ax, conj_a, conj_b)
        (c,), _ = self._run(key, lambda p, t: [p.tensordot(t[0], t[1], ax, conj_a=conj_a, conj_b=conj_b)], [a, b])
        return c

    def scale(self, a, s):
        a = self._c(a)
        out = self.tensordot(a.reshape(-1, 1), np.array([[s]], dtype=np.complex128), ([1], [0]))
        return out.reshape(a.shape)

    def lincomb(self, a, alpha, b, beta):
        """alpha a + beta b as one GEMM  [a | b] [[alpha I], [beta I]]."""
        a, b = self._c(a), self._c(b)
        shape = a.shape
        a2, b2 = a.reshape(-1, shape[-1]), b.reshape(-1, shape[-1])
        r, c = a2.shape
        coef = np.concatenate([alpha * np.eye(c), beta * np.eye(c)], axis=0).astype(np.complex128)

        def build(p, t):
            z = p.zeros((r, 1, 2 * c))
            p.embed(z, (0, 0, 0), t[0].reshape(r, 1, c))
            p.embed(z, (0, 0, c), t[1].reshape(r, 1, c))
            return [p.matmul(z.reshape(r, 2 * c), t[2], r, c, 2 * c)]
        (out,), _ = self._run(("lc", r, c), build, [a2, b2, coef])
        return out.reshape(shape)

    def hermitize(self, m):
        m = self._c(m)
        return self.lincomb(m, 0.5, np.conj(m.T), 0.5)

    def norm(self, a) -> float:
        a = self._c(a).reshape(-1)
        if a.size == 0:
            return 0.0

        def build(p, t):
            x = p.copy(t[0])
            p.normalize_(x, 0)
            return [x]
        _, sl = self._run(("nrm", a.size), build, [a])
        v = float(sl[0])
        return math.exp(v) if np.isfinite(v) and v != 0.0 else float(np.linalg.norm(a) == 0.0 and 0.0 or math.exp(v))

    def qr(self, m):
        m = self._c(m)
        (q, r), _ = self._run(("qr", m.shape), lambda p, t: list(p.qr(t[0])), [m])
        return q, r

    def _svd_raw(self, m):
        m = self._c(m)
        k = min(m.shape)

        def build(p, t):
            us, vh = p.svd_trunc(t[0], k, False, 0, 1)
            g = p.matmul(us, us, k, k, m.shape[0], 2, 0)            # US^H US: its diagonal holds s^2
            return [us, vh, g]
        (us, vh, g), _ = self._run(("svd", m.shape), build, [m])
        s = np.sqrt(np.maximum(np.real(np.diag(g)), 0.0))
        return us, s, vh

    def svd(self, m):
        us, s, vh = self._svd_raw(m)
        inv = np.where(s > 0, 1.0 / np.where(s > 0, s, 1.0), 0.0)
        u = self.tensordot(us, np.diag(inv).astype(np.complex128), ([1], [0]))
        return u, s, vh

    def eigh(self, h):
        """Hermitian eigen-decomposition, eigenvalues ascending: Jacobi SVD of the positive definite H / |H|_F + 1.5 I."""
        h = self._c(h)
        n = h.shape[0]
        nrm = self.norm(h)
        if not nrm > 0.0:
            return np.zeros(n), np.eye(n, dtype=np.complex128)
        m = self.lincomb(h, 1.0 / nrm, np.eye(n, dtype=np.complex128), _EIG_SHIFT)
        us, s, vh = self._svd_raw(m)
        w = (s - _EIG_SHIFT) * nrm
        order = np.argsort(w, kind="stable")
        return w[order], np.conj(vh[order]).T


# ------------------------------------------------------------------------------------------------
# resident executor: the same operations, but tensors stay in HBM between calls
# ------------------------------------------------------------------------------------------------
class RArr:
    """handle of a tensor that lives in the resident backend's arena.  Converting it to numpy (np.asarray, indexing)
    downloads it; the ITE algebra only does that for small tensors and for scalar decisions."""
    __slots__ = ("B", "dt")

    def __init__(self, B, dt):
        self.B, self.dt = B, dt

    shape = property(lambda self: self.dt.shape)
    ndim = property(lambda self: self.dt.ndim)
    size = property(lambda self: self.dt.size)

    def __array__(self, dtype=None, copy=None):
        a = self.B.to_host(self)
        return a if dtype is None else a.astype(dtype)

    def __getitem__(self, idx):
        return self.B.to_host(self)[idx]

    def copy(self):
        return self                      # tensors are never modified in place by the backend


class ResidentBackend:
    """device execution with a persistent arena: every call appends a few ops to one growing tensor program; the queued ops are
    launched (one kbp_run, asynchronous on the context's stream) only when the host needs a value -- ``to_host``, ``norm``, the
    singular values of ``svd`` / ``eigh`` -- or uploads one (``put``).  Buffers are recycled by the program's first-fit
    allocator when their Python handles die (all work is stream-ordered, so reuse is safe).  Host <-> device traffic is limited to the
    inputs (unit-cell tensors, ring tensors of the ToCore chains), small matrices built on the host (diag(sqrt(S)), ...)
    and the results that host code actually looks at."""

    def __init__(self, engine_key="ite-resident", device: int = 0, arena_elems: int | None = None):
        import os
        self.eng = get_engine(engine_key, device)
        if arena_elems is None:
            arena_elems = int(float(os.environ.get("KBP_ITE_ARENA_GB", "8")) * (1 << 30) / 16)
        self.arena_elems = arena_elems
        self.p = Program(8)
        self.eng.reserve(arena_elems, 1, 8)
        self.eng._loaded = None
        self.calls = 0

    # ---------------------------------------------------------------- plumbing
    def _flush(self):
        if self.p.words:
            if self.p.peak + 64 > self.arena_elems:
                raise MemoryError(f"resident ITE arena too small ({self.arena_elems} elements): set KBP_ITE_ARENA_GB")
            words, self.p.words = self.p.words, []      # a failing run must not leave its ops queued in front of the next call
            self.eng.run(np.array(words, dtype=np.int64))
            self.calls += 1

    def put(self, a) -> RArr:
        a = np.ascontiguousarray(a, dtype=np.complex128)
        self._flush()                                   # an upload must not overtake queued ops that still read a recycled buffer
        t = self.p.new(a.shape if a.ndim else (1,))
        if self.p.peak + 64 > self.arena_elems:
            raise MemoryError(f"resident ITE arena too small ({self.arena_elems} elements): set KBP_ITE_ARENA_GB")
        if a.size:
            self.eng.upload(t.off, a.reshape(-1), chain=0)
        return RArr(self, t)

    def _dt(self, x):
        return x.dt if isinstance(x, RArr) else self.put(x).dt

    def to_host(self, x: RArr) -> np.ndarray:
        self._flush()
        if x.size == 0:
            return np.zeros(x.shape, dtype=np.complex128)
        return self.eng.download(x.dt.off, x.size, chain=0).reshape(x.shape)

    # ---------------------------------------------------------------- data movement
    def reshape(self, a, shape):
        if not isinstance(a, RArr):
            return np.reshape(np.asarray(a), shape)
        shape = tuple(int(s) for s in (shape if not isinstance(shape, int) else (shape,)))
        if -1 in shape:
            known = int(np.prod([s for s in shape if s != -1]))
            shape = tuple(a.size // known if s == -1 else s for s in shape)
        return RArr(self, a.dt.reshape(shape))

    def transpose(self, a, perm):
        if not isinstance(a, RArr):
            return np.transpose(np.asarray(a), perm)
        return RArr(self, self.p.transpose(a.dt, perm))

    # ---------------------------------------------------------------- device ops
    def tensordot(self, a, b, axes, conj_a=False, conj_b=False):
        A, Bt = self._dt(a), self._dt(b)
        if isinstance(axes, int):
            assert axes == 0
            c = self.p.matmul(A.reshape(A.size, 1), Bt.reshape(1, Bt.size), A.size, Bt.size, 1, 3 if conj_a else 0, 3 if conj_b else 0)
            out = RArr(self, c.reshape(A.shape + Bt.shape))
        else:
            ax = (tuple(int(x) for x in axes[0]), tuple(int(x) for x in axes[1]))
            out = RArr(self, self.p.tensordot(A, Bt, ax, conj_a=conj_a, conj_b=conj_b))
        return out

    def scale(self, a, s):
        A = self._dt(a)
        c = self.p.matmul(A.reshape(A.size, 1), self.put(np.array([[s]], dtype=np.complex128)).dt, A.size, 1, 1)
        return RArr(self, c.reshape(A.shape))

    def lincomb(self, a, alpha, b, beta):
        A, Bt = self._dt(a), self._dt(b)
        shape = A.shape
        c = shape[-1]
        r = A.size // c
        coef = self.put(np.concatenate([alpha * np.eye(c), beta * np.eye(c)], axis=0))
        z = self.p.zeros((r, 1, 2 * c))
        self.p.embed(z, (0, 0, 0), A.reshape(r, 1, c))
        self.p.embed(z, (0, 0, c), Bt.reshape(r, 1, c))
        return RArr(self, self.p.matmul(z.reshape(r, 2 * c), coef.dt, r, c, 2 * c).reshape(shape))

    def hermitize(self, m):
        M = self._dt(m)
        mh = RArr(self, self.p.transpose(M, (1, 0), conj=True))
        return self.lincomb(RArr(self, M), 0.5, mh, 0.5)

    def norm(self, a) -> float:
        A = self._dt(a)
        if A.size == 0:
            return 0.0
        self._flush()
        self.eng.slots_zero()
        x = self.p.copy(A)
        self.p.normalize_(x, 0)
        self._flush()
        v = float(self.eng.slots()[0, 0])
        if v == 0.0:                       # |a| = 1 exactly or a = 0: tell them apart on the host (tiny)
            return float(np.linalg.norm(self.to_host(RArr(self, A))))
        return math.exp(v)

    def qr(self, m):
        M = self._dt(m)
        if os.environ.get("KBP_LINALG_DEBUG"):
            print(f"[kbp linalg] qr {M.shape}", flush=True)
        q, r = self.p.qr(M)
        return RArr(self, q), RArr(self, r)

    def _svd_raw(self, m):
        M = self._dt(m)
        k = min(M.shape)
        us, vh = self.p.svd_trunc(M, k, False, 0, 1)
        g = self.p.matmul(us, us, k, k, M.shape[0], 2, 0)
        self._flush()
        s = np.sqrt(np.maximum(np.real(np.diag(self.to_host(RArr(self, g)))), 0.0))
        if self.eng.slots()[0, -1] > 0:                 # engine status slot (include/kbp.h): the factorisation did not converge
            self.eng.slots_zero()
            raise BubbleConError(f"SVD of a {M.shape[0]} x {M.shape[1]} matrix did not converge on the device")
        return RArr(self, us), s, RArr(self, vh)

    def svd(self, m):
        us, s, vh = self._svd_raw(m)
        inv = np.where(s > 0, 1.0 / np.where(s > 0, s, 1.0), 0.0)
        return self.tensordot(us, np.diag(inv).astype(np.complex128), ([1], [0])), s, vh

    def eigh(self, h):
        H = self._dt(h)
        n = H.shape[0]
        nrm = self.norm(RArr(self, H))
        if not nrm > 0.0:
            return np.zeros(n), np.eye(n, dtype=np.complex128)
        m = self.lincomb(RArr(self, H), 1.0 / nrm, np.eye(n, dtype=np.complex128), _EIG_SHIFT)
        us, s, vh = self._svd_raw(m)
        w = (s - _EIG_SHIFT) * nrm
        order = np.argsort(w, kind="stable")
        return w[order], np.conj(self.to_host(vh)[order]).T


# ------------------------------------------------------------------------------------------------
# tracing backend: the same algebra recorded into one compiled program, no host values at all
# ------------------------------------------------------------------------------------------------
class TArr:
    """handle of a tensor recorded by a ``TraceBackend``: it has a shape but no value while the program is being built.
    Converting it to numpy or indexing it raises, so host code that would need a value fails when the program is compiled,
    not when it runs."""
    __slots__ = ("dt",)

    def __init__(self, dt):
        self.dt = dt

    shape = property(lambda self: self.dt.shape)
    ndim = property(lambda self: self.dt.ndim)
    size = property(lambda self: self.dt.size)

    def __array__(self, dtype=None, copy=None):
        raise TypeError(f"a traced tensor {self.shape} has no host value: the compiled program must not branch on data")

    def __getitem__(self, idx):
        raise TypeError(f"a traced tensor {self.shape} cannot be indexed on the host: reshape it through the backend")

    def copy(self):
        return self


class TraceBackend:
    """the backend interface of ``edge_env`` and ``ite.rho_ij_unnormalized`` (reshape, transpose, tensordot, qr) recorded into
    the ``Program`` ``p``.  Every operand must be a ``TArr`` of that program (inputs are declared by the caller); there are no
    scalar results, so nothing the trace does depends on data and the program replays for any batch of chains."""

    def __init__(self, p: Program):
        self.p = p

    @staticmethod
    def _dt(x):
        if not isinstance(x, TArr):
            raise TypeError(f"TraceBackend operand of type {type(x).__name__}: declare it as a program input")
        return x.dt

    def reshape(self, a, shape):
        A = self._dt(a)
        shape = tuple(int(s) for s in (shape if not isinstance(shape, int) else (shape,)))
        if -1 in shape:
            known = _prod(s for s in shape if s != -1)
            shape = tuple(A.size // known if s == -1 else s for s in shape)
        return TArr(A.reshape(shape))

    def transpose(self, a, perm):
        return TArr(self.p.transpose(self._dt(a), perm))

    def tensordot(self, a, b, axes, conj_a=False, conj_b=False):
        ax = (tuple(int(x) for x in axes[0]), tuple(int(x) for x in axes[1]))
        return TArr(self.p.tensordot(self._dt(a), self._dt(b), ax, conj_a=conj_a, conj_b=conj_b))

    def qr(self, m):
        q, r = self.p.qr(self._dt(m))
        return TArr(q), TArr(r)
