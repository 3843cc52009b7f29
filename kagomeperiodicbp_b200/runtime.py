"""Compiled tensor programs and their execution on an ``Engine``.

A ``Compiled`` program owns: the op stream, the packed input layout (all inputs are contiguous at the
bottom of the chain arena -> ONE host->device copy per run), the constant pool (identity sites,
uploaded once per load) and the packed output layout (outputs are gathered into one contiguous block
by the last ops of the program -> ONE device->host copy per run).
"""
from __future__ import annotations

import threading

import numpy as np

from .engine import E_SVD_NOCONV, Engine
from .program import ALIGN, DT, Program, _prod


class Compiled:
    def __init__(self, prog: Program, inputs: list, outputs: list, meta=None):
        """inputs: [(name, DT)] in declaration order (must be the first allocations of ``prog``);
        outputs: [(name, DT)]."""
        self.prog = prog
        self.in_layout = [(name, t.off, t.shape) for name, t in inputs]
        self.in_elems = max([t.off + t.size for _, t in inputs], default=0)
        # gather outputs
        pos, lay = 0, []
        for name, t in outputs:
            lay.append((name, pos, t.shape))
            pos += (t.size + ALIGN - 1) // ALIGN * ALIGN
        self.out_elems = max(pos, ALIGN)
        self.out_block = prog.new((self.out_elems,), pinned=True)
        for (name, t), (_, q, _) in zip(outputs, lay):
            if t.size:
                prog._emit(1, self.out_block.off + q, t.off, 0, 1, t.size, 0)   # OP_PERMUTE as a flat copy
        self.out_layout = lay
        self.words = prog.finalize()
        self.arena_elems = prog.arena_elems
        self.n_slots = prog.n_slots
        self.meta = meta or {}
        self.flops = prog.flops

    # -------------------------------------------------------------------------------------------
    def load(self, eng: Engine, nb: int):
        if getattr(eng, "_loaded", None) is self and eng.nb == nb:
            eng.slots_zero()
            return
        eng.reserve(self.arena_elems, nb, self.n_slots)
        for t, arr in self.prog.consts:
            eng.broadcast(t.off, arr)
        eng._loaded = self

    def pack_inputs(self, batch: list) -> np.ndarray:
        """batch: list (one per chain) of {name: ndarray}."""
        buf = np.zeros((len(batch), max(self.in_elems, 1)), dtype=np.complex128)
        for c, d in enumerate(batch):
            for name, off, shape in self.in_layout:
                a = np.asarray(d[name])
                assert tuple(a.shape) == tuple(shape) or a.size == _prod(shape), (name, a.shape, shape)
                buf[c, off:off + a.size] = a.reshape(-1)
        return buf

    def launch(self, eng: Engine, batch: list, soft_errors=()):
        """first half of ``run``: load, ONE host->device copy of the packed inputs, start the program.  Returns rc.  When the
        engine holds this program as a CUDA graph (``eng.graph_ready(self.words)``) the call returns as soon as the graph
        launch is queued: several engines can be started back to back from one host thread."""
        self.load(eng, len(batch))
        eng.upload(0, self.pack_inputs(batch))
        return eng.run(self.words, soft_errors=soft_errors)

    def collect(self, eng: Engine, nb: int, rc: int = 0):
        """second half of ``run``: ONE device->host copy of the packed outputs + the slot table (waits for the program)."""
        raw = eng.download(self.out_block.off, self.out_elems)
        slots = eng.slots()
        if rc == 0 and slots.shape[1] and np.any(slots[:, -1] > 0):     # engine-reserved status slot (include/kbp.h)
            rc = E_SVD_NOCONV
        outs = []
        for c in range(nb):
            d = {}
            for name, q, shape in self.out_layout:
                n = _prod(shape)
                d[name] = raw[c, q:q + n].reshape(shape).copy()
            outs.append(d)
        return outs, slots, rc

    def run(self, eng: Engine, batch: list, soft_errors=()):
        """returns (list of {name: ndarray} per chain, slots[nb, n_slots], rc)."""
        rc = self.launch(eng, batch, soft_errors=soft_errors)
        return self.collect(eng, len(batch), rc)

    # device-resident variant used by the benchmark: inputs already uploaded, outputs left on the device
    def run_resident(self, eng: Engine, soft_errors=()):
        eng.slots_zero()
        return eng.run(self.words, soft_errors=soft_errors)

    def verify_resident(self, eng: Engine, soft_errors=()) -> bool:
        """returns False (no rerun needed) and touches nothing: bench.py calls it after every ``run_resident``."""
        return False


_tls = threading.local()
_engines_lock = threading.Lock()
_engines: dict = {}


def get_engine(key="default", device: int = 0) -> Engine:
    """process-wide pool of engines (one CUDA stream + arena each), keyed by an arbitrary label so that
    e.g. the six block sides run on six concurrent streams."""
    with _engines_lock:
        k = (key, device)
        if k not in _engines:
            _engines[k] = Engine(device)
        return _engines[k]


def close_engines():
    with _engines_lock:
        for e in _engines.values():
            e.close()
        _engines.clear()
