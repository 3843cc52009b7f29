"""TEST INFRASTRUCTURE: a numpy interpreter for the tensor-program op stream (include/kbp.h).

It lets the CPU-only test tier validate everything on the host side of the C ABI -- program
compilation, buffer lifetimes / aliasing in the arena, slot bookkeeping, the packed input/output
layouts -- against the oracle, without a GPU.  The product never imports this file; on a GPU box the
same programs run through libkbp.so and are compared with the same oracle.
"""
from __future__ import annotations

import math
import struct

import numpy as np

from kagomeperiodicbp_b200.engine import (OP_EMBED, OP_EYE, OP_GEMM, OP_NONFINITE, OP_NORMALIZE, OP_PERMUTE, OP_QR,
                                          OP_SCALAR_TO_SLOT, OP_SVD, OP_ZERO)
from kagomeperiodicbp_b200.program import _prod


def _op(a, rows, cols, op):
    """matrix op(M) of shape rows x cols from flat storage."""
    if op in (0, 3):
        m = a[:rows * cols].reshape(rows, cols)
    else:
        m = a[:rows * cols].reshape(cols, rows).T
    if op in (2, 3):
        m = np.conj(m)
    return m


class NumpyEngine:
    """duck-types kagomeperiodicbp_b200.engine.Engine"""

    svd_input_norms = None               # a list: every OP_SVD appends the Frobenius norm of its input (input norm survey)

    def __init__(self):
        self.nb = 0
        self.n_slots = 0
        self.arena = None
        self._slots = None
        self._launches = 0

    def reserve(self, chain_elems, nb, n_slots=16):
        self.arena = np.full((nb, int(chain_elems)), np.nan + 1j * np.nan, dtype=np.complex128)
        self._slots = np.zeros((nb, n_slots))
        self.nb, self.n_slots = nb, n_slots

    def upload(self, offset, arr, chain=-1):
        a = np.asarray(arr, dtype=np.complex128)
        if chain < 0:
            self.arena[:, offset:offset + a.shape[1]] = a
        else:
            self.arena[chain, offset:offset + a.size] = a.ravel()

    def broadcast(self, offset, arr):
        a = np.asarray(arr, dtype=np.complex128).ravel()
        self.arena[:, offset:offset + a.size] = a[None, :]

    def download(self, offset, n, chain=-1):
        return self.arena[:, offset:offset + n].copy() if chain < 0 else self.arena[chain, offset:offset + n].copy()

    def slots(self):
        return self._slots.copy()

    def slots_zero(self):
        self._slots[:] = 0

    # zero-copy views, as Engine's (torch CPU tensors sharing the interpreter's memory)
    def arena_tensor(self):
        import torch
        return torch.from_numpy(self.arena.reshape(-1))

    def slots_tensor(self):
        import torch
        return torch.from_numpy(self._slots.reshape(-1))

    def torch_stream(self):
        return None

    def graph_ready(self, words):
        return True                      # the interpreter never blocks: exercises the one-thread launch / collect path

    def sync(self):
        pass

    def gemm_flops(self):
        return 0.0

    def launch_count(self):
        return self._launches

    def run(self, words, soft_errors=()):
        w = [int(x) for x in words]
        for c in range(self.nb):
            self._run_chain(w, self.arena[c], self._slots[c])
        return 0

    def _run_chain(self, w, ar, sl):
        i = 0
        while i < len(w):
            op = w[i]
            self._launches += 1
            if op == OP_PERMUTE:
                dst, src, cj, nd = w[i + 1:i + 5]
                dims = w[i + 5:i + 5 + nd]
                perm = w[i + 5 + nd:i + 5 + 2 * nd]
                n = _prod(dims)
                x = ar[src:src + n].reshape(dims).transpose(perm)
                if cj:
                    x = np.conj(x)
                ar[dst:dst + n] = np.ascontiguousarray(x).ravel()
                i += 5 + 2 * nd
            elif op == OP_GEMM:
                C, A, B, m, n, k, oa, ob = w[i + 1:i + 9]
                a = _op(ar[A:A + m * k], m, k, oa)
                b = _op(ar[B:B + k * n], k, n, ob)
                ar[C:C + m * n] = (a @ b).ravel()
                i += 9
            elif op == OP_QR:
                A, Q, R, wk, m, n = w[i + 1:i + 7]
                q, r = np.linalg.qr(ar[A:A + m * n].reshape(m, n))
                kk = min(m, n)
                ar[Q:Q + m * kk] = q.ravel()
                ar[R:R + kk * n] = r.ravel()
                i += 7
            elif op == OP_SVD:
                A, US, Vh, wk, m, n, keep, nrb, s0, s1, warm = w[i + 1:i + 12]
                u, s, vh = np.linalg.svd(ar[A:A + m * n].reshape(m, n), full_matrices=False)
                fro = np.linalg.norm(s)
                if NumpyEngine.svd_input_norms is not None:
                    NumpyEngine.svd_input_norms.append(float(fro))
                if s1 >= 0 and fro > 0:
                    sl[s1] += math.sqrt(np.sum(s[keep:] ** 2) / np.sum(s ** 2))
                if nrb and fro > 0:
                    s = s / fro
                    if s0 >= 0:
                        sl[s0] += math.log(fro)
                ar[US:US + m * keep] = (u[:, :keep] * s[:keep]).ravel()
                ar[Vh:Vh + keep * n] = vh[:keep].ravel()
                ar[wk:wk + 1] = np.nan  # scratch is clobbered
                i += 12
            elif op == OP_NORMALIZE:
                buf, n, slot = w[i + 1:i + 4]
                nr = np.linalg.norm(ar[buf:buf + n])
                if nr > 0:
                    ar[buf:buf + n] /= nr
                    if slot >= 0:
                        sl[slot] += math.log(nr)
                i += 4
            elif op == OP_EMBED:
                dst, src, arb, aib, d0, d1, d2, s0, s1, s2, ss = w[i + 1:i + 12]
                alpha = complex(*struct.unpack("dd", struct.pack("qq", arb, aib)))
                if ss >= 0:
                    alpha *= 1.0 if sl[ss] > 0 else -1.0
                x = ar[src:src + d0 * d1 * d2].reshape(d0, d1, d2)
                idx = (np.arange(d0)[:, None, None] * s0 + np.arange(d1)[None, :, None] * s1 + np.arange(d2)[None, None, :] * s2)
                ar[dst + idx] = alpha * x
                i += 12
            elif op == OP_ZERO:
                dst, n = w[i + 1:i + 3]
                ar[dst:dst + n] = 0
                i += 3
            elif op == OP_SCALAR_TO_SLOT:
                buf, sre, sim = w[i + 1:i + 4]
                if sre >= 0:
                    sl[sre] = ar[buf].real
                if sim >= 0:
                    sl[sim] = ar[buf].imag
                i += 4
            elif op == OP_NONFINITE:
                buf, n, slot = w[i + 1:i + 4]
                sl[slot] += np.sum(~np.isfinite(ar[buf:buf + n]))
                i += 4
            elif op == OP_EYE:
                dst, r, c = w[i + 1:i + 4]
                ar[dst:dst + r * c] = np.eye(r, c).ravel()
                i += 4
            else:
                raise ValueError(f"unknown opcode {op} at word {i}")
