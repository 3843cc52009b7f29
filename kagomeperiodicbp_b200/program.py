"""Tensor-program builder: records numpy-style operations on *device tensors* (static shapes) as the
flat int64 op stream ``kbp_run`` executes (include/kbp.h).  Nothing here touches data: a program is
compiled once per shape signature, cached, and replayed with fresh inputs.

Buffers live in one arena per chain; offsets are assigned at build time by a first-fit allocator
driven by the Python lifetime of the ``DT`` handles (CPython refcounting makes this deterministic),
so a replay needs no allocation at all.
"""
from __future__ import annotations

import struct

import numpy as np

from .engine import (OP_EMBED, OP_EYE, OP_GEMM, OP_NONFINITE, OP_NORMALIZE, OP_PERMUTE, OP_QR, OP_SCALAR_TO_SLOT, OP_SU,
                     OP_SVD, OP_ZERO, qr_work_elems, svd_work_elems)

ALIGN = 8  # complex128 elements (128 B)


def _prod(s):
    r = 1
    for x in s:
        r *= int(x)
    return r


class _Block:
    __slots__ = ("prog", "off", "size", "pinned")

    def __init__(self, prog, off, size, pinned=False):
        self.prog, self.off, self.size, self.pinned = prog, off, size, pinned

    def __del__(self):
        try:
            if not self.pinned and self.prog is not None:
                self.prog._free(self.off, self.size)
        except Exception:
            pass


class DT:
    """device tensor handle: a contiguous row-major view of an arena block."""
    __slots__ = ("block", "shape")

    def __init__(self, block: _Block, shape):
        self.block = block
        self.shape = tuple(int(s) for s in shape)

    @property
    def off(self):
        return self.block.off

    @property
    def size(self):
        return _prod(self.shape)

    @property
    def ndim(self):
        return len(self.shape)

    def reshape(self, *shape):
        if len(shape) == 1 and isinstance(shape[0], (tuple, list)):
            shape = tuple(shape[0])
        assert _prod(shape) == self.size, (shape, self.shape)
        return DT(self.block, shape)


class Program:
    def __init__(self, n_slots: int = 16):
        self.words: list[int] = []
        self.top = 0
        self.peak = 0
        self.free: list[list[int]] = []      # sorted [off, size]
        self.inputs: dict[str, DT] = {}
        self.outputs: dict[str, DT] = {}
        self.consts: list[tuple[DT, np.ndarray]] = []
        self._const_cache: dict = {}
        self.n_slots = n_slots
        self.n_ops = 0
        self.flops = 0.0                      # algorithmic flops per chain (SURVEY section 8d conventions)
        self.svd_shapes: list[tuple[int, int, int]] = []
        self.qr_shapes: list[tuple[int, int]] = []
        self.gemm_flops = 0.0
        self._frozen = None

    # ---------------- allocation ----------------
    def _alloc_raw(self, n: int) -> int:
        n = max(ALIGN, (int(n) + ALIGN - 1) // ALIGN * ALIGN)
        for k, (off, size) in enumerate(self.free):
            if size >= n:
                if size == n:
                    self.free.pop(k)
                else:
                    self.free[k] = [off + n, size - n]
                return off
        off = self.top
        self.top += n
        self.peak = max(self.peak, self.top)
        return off

    def _free(self, off: int, n: int):
        n = max(ALIGN, (int(n) + ALIGN - 1) // ALIGN * ALIGN)
        fl = self.free
        lo, hi = 0, len(fl)
        while lo < hi:
            mid = (lo + hi) // 2
            if fl[mid][0] < off:
                lo = mid + 1
            else:
                hi = mid
        fl.insert(lo, [off, n])
        if lo + 1 < len(fl) and fl[lo][0] + fl[lo][1] == fl[lo + 1][0]:
            fl[lo][1] += fl[lo + 1][1]
            fl.pop(lo + 1)
        if lo > 0 and fl[lo - 1][0] + fl[lo - 1][1] == fl[lo][0]:
            fl[lo - 1][1] += fl[lo][1]
            fl.pop(lo)
            lo -= 1
        if fl and fl[-1][0] + fl[-1][1] == self.top:
            self.top = fl[-1][0]
            fl.pop()

    def new(self, shape, pinned=False) -> DT:
        n = _prod(shape)
        return DT(_Block(self, self._alloc_raw(n), n, pinned), shape)

    # ---------------- declarations ----------------
    def input(self, name: str, shape) -> DT:
        t = self.new(shape, pinned=True)
        self.inputs[name] = t
        return t

    def output(self, name: str, t: DT):
        t.block.pinned = True
        self.outputs[name] = t

    def const(self, arr: np.ndarray) -> DT:
        a = np.ascontiguousarray(arr, dtype=np.complex128)
        key = (a.shape, a.tobytes())
        if key not in self._const_cache:
            t = self.new(a.shape, pinned=True)
            self.consts.append((t, a))
            self._const_cache[key] = t
        return self._const_cache[key]

    def _emit(self, *w):
        self.words.extend(int(x) for x in w)
        self.n_ops += 1

    # ---------------- ops ----------------
    def transpose(self, x: DT, perm, conj=False) -> DT:
        perm = [int(p) for p in perm]
        if perm == list(range(x.ndim)) and not conj:
            return x
        # drop size-1 axes and merge runs so the kernel sees <= 8 dims
        out_shape = [x.shape[p] for p in perm]
        dims = list(x.shape)
        keep = [i for i in range(len(dims)) if dims[i] != 1]
        if not keep:
            keep = [0]
        remap = {ax: k for k, ax in enumerate(keep)}
        p2 = [remap[p] for p in perm if p in remap]
        d2 = [dims[i] for i in keep]
        # merge axes adjacent both in source and destination
        groups = []
        for p in p2:
            if groups and groups[-1][-1] + 1 == p:
                groups[-1].append(p)
            else:
                groups.append([p])
        order = sorted(range(len(groups)), key=lambda g: groups[g][0])
        src_dims = [_prod(d2[a] for a in groups[g]) for g in order]
        pos = {g: k for k, g in enumerate(order)}
        perm3 = [pos[g] for g in range(len(groups))]
        assert len(src_dims) <= 8, "permute supports at most 8 merged axes"
        y = self.new(out_shape)
        self._emit(OP_PERMUTE, y.off, x.off, 1 if conj else 0, len(src_dims), *src_dims, *perm3)
        return y

    def copy(self, x: DT) -> DT:
        y = self.new(x.shape)
        self._emit(OP_PERMUTE, y.off, x.off, 0, 1, x.size, 0)
        return y

    def conj(self, x: DT) -> DT:
        y = self.new(x.shape)
        self._emit(OP_PERMUTE, y.off, x.off, 1, 1, x.size, 0)
        return y

    def matmul(self, a: DT, b: DT, m, n, k, opA=0, opB=0) -> DT:
        c = self.new((m, n))
        self._emit(OP_GEMM, c.off, a.off, b.off, m, n, k, opA, opB)
        self.flops += 8.0 * m * n * k
        self.gemm_flops += 8.0 * m * n * k
        return c

    def tensordot(self, a: DT, b: DT, axes, conj_a=False, conj_b=False) -> DT:
        ca, cb = [int(x) for x in axes[0]], [int(x) for x in axes[1]]
        fa = [i for i in range(a.ndim) if i not in ca]
        fb = [i for i in range(b.ndim) if i not in cb]
        M = _prod(a.shape[i] for i in fa)
        N = _prod(b.shape[i] for i in fb)
        K = _prod(a.shape[i] for i in ca)
        assert K == _prod(b.shape[i] for i in cb), (a.shape, b.shape, axes)
        # A operand
        if fa + ca == list(range(a.ndim)):
            A, opA = a, (3 if conj_a else 0)
        elif ca + fa == list(range(a.ndim)):
            A, opA = a, (2 if conj_a else 1)
        else:
            A, opA = self.transpose(a, fa + ca, conj=conj_a), 0
        if cb + fb == list(range(b.ndim)):
            B, opB = b, (3 if conj_b else 0)
        elif fb + cb == list(range(b.ndim)):
            B, opB = b, (2 if conj_b else 1)
        else:
            B, opB = self.transpose(b, cb + fb, conj=conj_b), 0
        c = self.matmul(A, B, M, N, K, opA, opB)
        return c.reshape([a.shape[i] for i in fa] + [b.shape[i] for i in fb])

    def qr(self, x: DT):
        m, n = x.shape
        k = min(m, n)
        q, r = self.new((m, k)), self.new((k, n))
        work = self.new((qr_work_elems(m, n),))
        self._emit(OP_QR, x.off, q.off, r.off, work.off, m, n)
        mm, nn = max(m, n), min(m, n)
        self.flops += 4.0 * (4.0 * mm * nn * nn - 4.0 * nn ** 3 / 3.0)
        self.qr_shapes.append((m, n))
        return q, r

    def lq(self, x: DT):
        """x (m x n) = L (m x k) Q (k x n), Q Q^H = I  -- the role scipy.linalg.rq(mode='economic') plays."""
        xh = self.transpose(x, (1, 0), conj=True)
        q, r = self.qr(xh)
        return self.transpose(r, (1, 0), conj=True), self.transpose(q, (1, 0), conj=True)

    def svd_trunc(self, x: DT, keep: int, nr_bulk: bool, slot_lognorm: int, slot_trunc: int):
        """rank-`keep` truncated SVD (the last op word is reserved)."""
        m, n = x.shape
        us, vh = self.new((m, keep)), self.new((keep, n))
        work = self.new((svd_work_elems(m, n),))
        self._emit(OP_SVD, x.off, us.off, vh.off, work.off, m, n, keep, 1 if nr_bulk else 0, slot_lognorm, slot_trunc, -1)
        mm, nn = max(m, n), min(m, n)
        self.flops += 4.0 * (14.0 * mm * nn * nn + 8.0 * nn ** 3)
        self.svd_shapes.append((m, n, keep))
        return us, vh

    def normalize_(self, x: DT, slot: int):
        """in place: x /= |x|, slot += ln|x|.  Caller guarantees x is not aliased."""
        self._emit(OP_NORMALIZE, x.off, x.size, slot)

    def zeros(self, shape) -> DT:
        t = self.new(shape)
        self._emit(OP_ZERO, t.off, t.size)
        return t

    def eye(self, rows: int, cols: int) -> DT:
        t = self.new((rows, cols))
        self._emit(OP_EYE, t.off, rows, cols)
        return t

    def embed(self, dst: DT, dst_index, src: DT, alpha=1.0, sign_slot=-1):
        """dst[i0 + i, j0 + j, k0 + k] = alpha * src[i, j, k]  (dst, src 3-D)."""
        assert dst.ndim == 3 and src.ndim == 3
        s0, s1, s2 = dst.shape[1] * dst.shape[2], dst.shape[2], 1
        off = dst.off + dst_index[0] * s0 + dst_index[1] * s1 + dst_index[2] * s2
        ar, ai = struct.unpack("qq", struct.pack("dd", float(np.real(alpha)), float(np.imag(alpha))))
        self._emit(OP_EMBED, off, src.off, ar, ai, *src.shape, s0, s1, s2, sign_slot)

    def scalar_to_slot(self, x: DT, slot_re: int, slot_im: int):
        self._emit(OP_SCALAR_TO_SLOT, x.off, slot_re, slot_im)

    def nonfinite(self, x: DT, slot: int):
        self._emit(OP_NONFINITE, x.off, x.size, slot)

    def simple_update_(self, gammas, lam: DT, gate: DT, rdm: DT, max_steps: int, tol: float, slots, bonds):
        """in place: up to ``max_steps`` simple-update steps of the unit cell (Gamma_A, Gamma_B, Gamma_C = ``gammas``, lambda
        [6, D]) with the two-site gate [d, d, d, d]; writes the six SU-environment RDMs to ``rdm`` [6, d, d, d, d].  ``slots``:
        (steps done, last step delta, non-finite entries); ``bonds``: six (site_i, leg_i, site_j, leg_j)."""
        d, D = gammas[0].shape[0], gammas[0].shape[1]
        (tol_bits,) = struct.unpack("q", struct.pack("d", float(tol)))
        self._emit(OP_SU, *(t.off for t in gammas), lam.off, gate.off, rdm.off, d, D, int(max_steps), tol_bits, *slots,
                   *(x for bond in bonds for x in bond))

    # ---------------- finish ----------------
    def finalize(self):
        if self._frozen is None:
            self._frozen = np.array(self.words, dtype=np.int64)
        return self._frozen

    @property
    def arena_elems(self) -> int:
        return self.peak + ALIGN
