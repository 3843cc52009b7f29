"""The ITE step on the device: one loop body of the reference's ``ite_per_mode``
(src/algo/imaginary_time_evolution/main.py:566-590) --

    robust_belief_propagation (warm messages)              -> belief_propagation.py (six device chains per iteration)
    reduce_tn(full_tn, ModeTN) / reduce_tn(mode_tn, EdgeTN) -> two device ToCore chains + edge_env.edge_environment
    ite_update_unit_cell (_tn_update.py:165-205)            -> ite.rho_ij / ite.apply_2local_gate on the device backend

and the energy measurement ``measure_energies_and_observables_together`` (src/algo/measurements.py:163-243: six edge RDMs of
one mode, energy per site = sum / 3).  Host code orchestrates and moves data; all tensor algebra runs through libkbp.so.
``measure_energies_batch`` measures many unit cells at once: the reduction after the ToCore chains is shape-only, so it is
compiled once (``compile_measurement``, recorded through ``linalg.TraceBackend``) and launched with one chain per cell.
The core is reduced with bottom-up direction U unless told otherwise (the reference draws it at random from {U, DL, DR},
kagome_to_core.py:178-179; SURVEY 8d fixes U for reproducible runs; `reduce_to_core(..., direction=)` takes all three).
"""
from __future__ import annotations

import time
from dataclasses import dataclass, field

import numpy as np

from . import belief_propagation as bp
from . import edge_env, ite, linalg
from .bubblecon import bubblecon as device_bubblecon
from .containers import BPConfig, UnitCell
from .dev_bubblecon import trace_bubblecon
from .dev_mps import SLOT_NONFINITE
from .engine import E_SVD_NOCONV, BubbleConError
from .lattice import BLOCK_SIDES_CCW
from .linalg import ResidentBackend, TArr, TraceBackend
from .program import Program
from .runtime import Compiled, get_engine

_backend = None


def backend() -> ResidentBackend:
    global _backend
    if _backend is None:
        _backend = ResidentBackend("ite")
    return _backend


def _device_bubblecon_fn(T_list, edges, angles, bubble_angle, order, chi, kets):
    mp = device_bubblecon([np.ascontiguousarray(np.asarray(t), dtype=np.complex128) for t in T_list], edges, angles, bubble_angle, order,
                          D_trunc=chi, ket_tensors=kets, engine_key="ite-bubblecon")
    return mp.A


def reduce_to_core(unit_cell: UnitCell, messages: dict, N: int, chi: int, device: int = 0, direction: str = "U"):
    """the 12 ring tensors of the CoreTN (kagome_to_core.py:322-364): two truncated ToCore chains (bottom-up ``direction`` in
    {U, DL, DR} and its opposite) run concurrently on two streams, then the overlap zip on the device backend."""
    bu_side, td_side, _ = edge_env.CORE_DIRECTIONS[direction]
    d, D = unit_cell.A.shape[0], unit_cell.A.shape[1]
    shapes = bp._msg_shapes(messages)
    futs = []
    for side in (bu_side, td_side):
        comp = bp.compile_side_program(N, d, D, side, chi, shapes, None, depth="ToCore", epilogue=False, arbitrary=bp._is_arbitrary(unit_cell))
        batch = [bp._side_inputs(unit_cell, messages, comp)]
        futs.append(bp._pool.submit(bp._run_side, side, comp, batch, device))
    res = {}
    for f in futs:
        side, outs, slots, rc = f.result()
        bp.raise_if_not_converged(rc, f"ToCore contraction towards {side}")
        if slots[0, bp.SLOT_NONFINITE] > 0:
            raise bp.BubbleConError(f"non-finite values in the ToCore contraction towards {side}")
        o = outs[0]
        res[side] = [o[f"out{k}"] for k in range(len(o))]
    return edge_env.core_env_tensors(backend(), N, res[bu_side], res[td_side], direction)


def edge_tn(unit_cell: UnitCell, env12, N: int, mode: str, edge: str, chi: int):
    """(Ti, Tj, mps_env, info) of the EdgeTN in canonical order (reduce_core_to_mode + reduce_mode_to_edge)."""
    return edge_env.edge_environment(backend(), N, unit_cell.tensors(), env12, mode, edge, chi, _device_bubblecon_fn)


_PAULI = {"x": np.array([[0, 1], [1, 0]], dtype=np.complex128), "y": np.array([[0, -1j], [1j, 0]], dtype=np.complex128),
          "z": np.array([[1, 0], [0, -1]], dtype=np.complex128)}


def expectation_values_with_rdm(rdm) -> dict:
    """(src/algo/measurements.py:522-545)  {pauli: (<sigma> on site i, <sigma> on site j)} from the one-site marginals of a
    two-site RDM rho[i, i*, j, j*] -- 2 x 2 host arithmetic, as in the reference."""
    rho_i = np.trace(rdm, axis1=2, axis2=3)
    rho_j = np.trace(rdm, axis1=0, axis2=1)
    return {k: (float(np.real(np.trace(s @ rho_i))), float(np.real(np.trace(s @ rho_j)))) for k, s in _PAULI.items()}


def negativity_of_rdm(rdm) -> float:
    """(src/algo/measurements.py:91-94, src/physics/metrics/_negativity.py:43-73)  sum of |negative eigenvalues| of the partial
    transpose (first site) of the 4 x 4 two-site density matrix."""
    pt = np.transpose(rdm, (1, 0, 2, 3))                               # i <-> i*
    mat = np.transpose(pt, (0, 2, 1, 3)).reshape(4, 4)
    w = np.linalg.eigvals(mat)
    return float(sum(abs(x) for x in w if x.real < 0))


@dataclass
class MeasurementsOnUnitCell:
    """(src/containers/results.py:8-30)"""
    energies: dict
    rdms: dict = field(default_factory=dict)
    expectations: dict = field(default_factory=dict)      # {A|B|C: {x|y|z: mean over the edges the site appears on}}
    entanglement: dict = field(default_factory=dict)      # negativity per edge

    @property
    def mean_energy(self) -> float:
        return sum(self.energies.values()) / 3

    @property
    def mean_expectation_values(self) -> dict:
        return {k: sum(self.expectations[f][k] for f in "ABC") / 3 for k in "xyz"}


def measurements_from_rdms(rdms: dict, flavors: dict, h) -> MeasurementsOnUnitCell:
    """the host end of a measurement: energy, <sigma> and negativity of every edge from its trace-normalised two-site RDM.
    ``rdms`` / ``flavors``: {edge: rho[i, i*, j, j*]} / {edge: (flavour of site i, flavour of site j)} in ``edge_env.EDGES``
    order.  4 x 4 host arithmetic, as in the reference."""
    energies, ent = {}, {}
    acc = {f: {k: [0.0, 0] for k in "xyz"} for f in "ABC"}
    for e, rho in rdms.items():
        key = f"({e[0]}, {e[1]})"
        energies[key] = float(np.real(np.dot(np.asarray(rho).flatten(), h.flatten())))
        ent[key] = negativity_of_rdm(rho)
        for k, vals in expectation_values_with_rdm(rho).items():
            for v, f in zip(vals, flavors[e]):
                acc[f][k][0] += v
                acc[f][k][1] += 1
    expectations = {f: {k: (acc[f][k][0] / acc[f][k][1] if acc[f][k][1] else 0.0) for k in "xyz"} for f in "ABC"}
    return MeasurementsOnUnitCell(energies, dict(rdms), expectations, ent)


def measure_energies(unit_cell: UnitCell, messages: dict, N: int, chi: int, h=None, mode: str = "A", env12=None) -> MeasurementsOnUnitCell:
    """(src/algo/measurements.py:163-243, energies part)"""
    h = ite.heisenberg_afm() if h is None else np.asarray(h)
    if env12 is None:
        env12 = reduce_to_core(unit_cell, messages, N, chi)
    B = backend()
    rdms, flavors = {}, {}
    for e in edge_env.EDGES:
        ti, tj, env, info = edge_tn(unit_cell, env12, N, mode, e, chi)
        rdms[e] = ite.rho_ij(B, ti, tj, env)
        flavors[e] = info["flavors"]
    return measurements_from_rdms(rdms, flavors, h)


# ------------------------------------------------------------------------------------------------
# the measurement of a batch of unit cells as one compiled program
# ------------------------------------------------------------------------------------------------
_measure_cache: dict = {}


def compile_measurement(N: int, d: int, D: int, chi: int, mode: str, direction: str, tocore_shapes) -> Compiled:
    """the whole measurement after the two ToCore chains as ONE program, compiled from shapes only: the zip of the two
    boundary MPSs into the 12 ring tensors (``edge_env.core_env_tensors``), then for each of the six edges the Core -> Mode ->
    Edge reduction (``edge_env.edge_environment``, its truncated ToEdge contractions recorded in place by ``trace_bubblecon``)
    and the unnormalised two-site RDM (``ite.rho_ij_unnormalized``).  Every control decision of that code is shape-only and
    the truncated SVDs decide per chain on the device, so one program serves any batch of cells.

    ``tocore_shapes``: (site shapes of the bottom-up ToCore MPS, site shapes of the top-down one) of ``direction``.
    Inputs: cellA, cellB, cellC [d, D, D, D, D], bu{k} and td{k} (the MPS sites).  Outputs: rho{k} [d, d, d, d] for the edges
    of ``edge_env.EDGES``; slot SLOT_NONFINITE counts non-finite RDM entries.  meta["flavors"]: the site flavours per edge."""
    bu_shapes, td_shapes = (tuple(tuple(int(x) for x in sh) for sh in side) for side in tocore_shapes)
    key = (N, d, D, chi, mode, direction, bu_shapes, td_shapes)
    if key in _measure_cache:
        return _measure_cache[key]
    p = Program(bp.N_SLOTS)
    ins = [(nm, p.input(nm, (d, D, D, D, D))) for nm in ("cellA", "cellB", "cellC")]
    ins += [(f"bu{k}", p.input(f"bu{k}", sh)) for k, sh in enumerate(bu_shapes)]
    ins += [(f"td{k}", p.input(f"td{k}", sh)) for k, sh in enumerate(td_shapes)]
    B = TraceBackend(p)
    t = {nm: TArr(dt) for nm, dt in ins}
    cell = (t["cellA"], t["cellB"], t["cellC"])
    env12 = edge_env.core_env_tensors(B, N, [t[f"bu{k}"] for k in range(len(bu_shapes))],
                                      [t[f"td{k}"] for k in range(len(td_shapes))], direction)

    def bubblecon_fn(T_list, edges, angles, bubble_angle, order, D_trunc, kets):
        # what compile_bubblecon records for the per-cell path, here inside the measurement program
        mp, _ = trace_bubblecon(p, [x.dt for x in T_list], edges, angles, bubble_angle, list(order), D_trunc, kets)
        return [TArr(x) for x in mp.dense_sites()]

    outs, flavors = [], {}
    for k, e in enumerate(edge_env.EDGES):
        ti, tj, env, info = edge_env.edge_environment(B, N, cell, env12, mode, e, chi, bubblecon_fn)
        rho = ite.rho_ij_unnormalized(B, ti, tj, env).dt
        p.nonfinite(rho, SLOT_NONFINITE)
        outs.append((f"rho{k}", rho))
        flavors[e] = info["flavors"]
    comp = Compiled(p, ins, outs, meta=dict(flavors=flavors))
    _measure_cache[key] = comp
    return comp


def _measure_engine(device: int):
    """the measurement program's own engine (stream + arena), from the pool the ITE backends use"""
    return linalg.get_engine("measure", device)


def _measure_chunk(cells, messages_list, index, N, chi, mode, direction, device):
    """rdms ({edge: trace-normalised rho}) and flavours of the cells ``index`` (one shape group, one launch each)."""
    bu_side, td_side, _ = edge_env.CORE_DIRECTIONS[direction]
    d, D = cells[index[0]].A.shape[0], cells[index[0]].A.shape[1]
    shapes = bp._msg_shapes(messages_list[index[0]])
    futs = []
    for side in (bu_side, td_side):
        comp = bp.compile_side_program(N, d, D, side, chi, shapes, None, depth="ToCore", epilogue=False)
        batch = [bp._side_inputs(cells[i], messages_list[i], comp) for i in index]
        futs.append(bp._pool.submit(bp._run_side, side, comp, batch, device))
    res = {}
    for f in futs:
        side, outs, slots, rc = f.result()
        for c, i in enumerate(index):
            if slots[c, -1] > 0:                   # engine status slot: a truncation of this chain did not converge
                raise BubbleConError(f"cell {i}: truncated SVD did not converge in the ToCore contraction towards {side}")
            if slots[c, bp.SLOT_NONFINITE] > 0:
                raise BubbleConError(f"cell {i}: non-finite values in the ToCore contraction towards {side}")
        res[side] = outs
    n_bu, n_td = len(res[bu_side][0]), len(res[td_side][0])
    comp = compile_measurement(N, d, D, chi, mode, direction,
                               ([res[bu_side][0][f"out{k}"].shape for k in range(n_bu)],
                                [res[td_side][0][f"out{k}"].shape for k in range(n_td)]))
    batch = []
    for c, i in enumerate(index):
        x = {"cellA": cells[i].A, "cellB": cells[i].B, "cellC": cells[i].C}
        x.update({f"bu{k}": res[bu_side][c][f"out{k}"] for k in range(n_bu)})
        x.update({f"td{k}": res[td_side][c][f"out{k}"] for k in range(n_td)})
        batch.append(x)
    outs, slots, rc = comp.run(_measure_engine(device), batch, soft_errors=(E_SVD_NOCONV,))
    rdms = []
    for c, i in enumerate(index):
        if slots[c, -1] > 0:
            raise BubbleConError(f"cell {i}: truncated SVD did not converge in a ToEdge contraction of the measurement")
        if slots[c, SLOT_NONFINITE] > 0:
            raise BubbleConError(f"cell {i}: non-finite values in the measurement")
        r = {}
        for k, e in enumerate(edge_env.EDGES):
            rho = outs[c][f"rho{k}"]
            r[e] = rho * (1.0 / ite.rho_trace(rho))          # the trace normalisation of ite.rho_ij, on the host
        rdms.append(r)
    return rdms, comp.meta["flavors"]


def measure_energies_batch(cells: list, messages_list: list, N: int, chi: int, h=None, mode: str = "A", direction: str = "U",
                           device: int = 0, batch: int = 8) -> list:
    """``measure_energies`` for a list of independent unit cells, ``batch`` cells per launch: cells with the same message
    shapes share the two ToCore chains (run concurrently on their side engines) and one launch of the compiled measurement
    program (``compile_measurement``); the host only normalises the RDMs and does the 4 x 4 arithmetic of every edge
    (``measurements_from_rdms``).  -> [MeasurementsOnUnitCell] in input order.

    Raises ValueError before any launch for an unknown ``mode`` / ``direction``, ``cells`` and ``messages_list`` of different
    lengths, a non-repeated block (``LatticeTensors``) or cells of different d / D; BubbleConError naming the cell for a
    truncation that did not converge or non-finite values."""
    if len(cells) != len(messages_list):
        raise ValueError(f"{len(cells)} cells but {len(messages_list)} message sets")
    if mode not in edge_env.MODES:
        raise ValueError(f"unknown mode {mode!r}: expected one of {edge_env.MODES}")
    if direction not in edge_env.CORE_DIRECTIONS:
        raise ValueError(f"unknown direction {direction!r}: expected one of {tuple(edge_env.CORE_DIRECTIONS)}")
    if batch < 1:
        raise ValueError(f"batch must be at least 1, got {batch}")
    if not cells:
        return []
    for i, c in enumerate(cells):
        if bp._is_arbitrary(c):
            raise ValueError(f"cell {i} is a non-repeated block (LatticeTensors): the batched measurement takes unit cells")
    d, D = cells[0].A.shape[0], cells[0].A.shape[1]
    for i, c in enumerate(cells):
        if any(t.shape != (d, D, D, D, D) for t in c.tensors()):
            raise ValueError(f"cell {i} has tensors of shapes {[t.shape for t in c.tensors()]}, cell 0 has d = {d}, D = {D}")
    h = ite.heisenberg_afm() if h is None else np.asarray(h)
    groups: dict = {}
    for i, m in enumerate(messages_list):
        groups.setdefault(bp._msg_shapes(m), []).append(i)
    out = [None] * len(cells)
    for idx in groups.values():
        for c0 in range(0, len(idx), batch):
            chunk = idx[c0:c0 + batch]
            rdms, flavors = _measure_chunk(cells, messages_list, chunk, N, chi, mode, direction, device)
            for i, r in zip(chunk, rdms):
                out[i] = measurements_from_rdms(r, flavors, h)
    return out


ENV_HERMICITY_THRESHOLD = 1e-4       # src/algo/imaginary_time_evolution/_constants.py
DEBUG_MODE = False                   # the reference's configuration.json "debug_mode": violations raise instead of warning


@dataclass
class MatrixMetrics:
    """(src/containers/density_matrices.py:5-13)"""
    eigenvalues: list
    negativity: float
    sum_eigenvalues: complex
    hermicity: float
    norm: float
    trace: complex
    other: dict = field(default_factory=dict)


def calc_metrics(rho: np.ndarray) -> MatrixMetrics:
    """(src/algo/density_matrices.py:31-42) of a d^2 x d^2 density matrix: 4 x 4 host arithmetic, as in the reference."""
    w = np.linalg.eigvals(rho)
    return MatrixMetrics(eigenvalues=list(w), negativity=float(sum(abs(np.real(v)) for v in w if np.real(v) < 0)),
                         sum_eigenvalues=complex(np.sum(w)), hermicity=float(np.linalg.norm(rho - np.conj(rho.T)) / np.linalg.norm(rho)),
                         norm=float(np.linalg.norm(rho)), trace=complex(np.trace(rho)))


def _raise_ite_error_or_print_warning(message: str):
    if DEBUG_MODE:
        raise ite.ITEError(message)
    import warnings
    warnings.warn(message, RuntimeWarning, stacklevel=3)


def check_rdms_metrics(rdm) -> MatrixMetrics:
    """the guard of every edge update (src/algo/imaginary_time_evolution/_tn_update.py:51-60): the two-site density matrix
    must be Hermitian to 1e-4, of unit trace (sum of eigenvalues) to 1e-4, and positive up to a total negativity of 0.1."""
    r = np.asarray(rdm)
    d = r.shape[0]
    m = calc_metrics(np.transpose(r, (0, 2, 1, 3)).reshape(d * d, d * d))          # rho_ij_to_rho (density_matrices.py:11-18)
    if m.hermicity > ENV_HERMICITY_THRESHOLD:
        _raise_ite_error_or_print_warning(f"env_hermicity={m.hermicity}")
    if abs(np.real(m.sum_eigenvalues) - 1) > ENV_HERMICITY_THRESHOLD:
        _raise_ite_error_or_print_warning(f"env is not psd. sum-eigenvalues={np.real(m.sum_eigenvalues)}")
    if m.negativity > 0.1:
        _raise_ite_error_or_print_warning(f"env is not psd. negativity={m.negativity}")
    return m


def _original_negativity_ratio(eigen_vals) -> float:
    """(_tn_update.py:63-73)"""
    if eigen_vals is None:
        return 0.0
    ev = np.real(np.asarray(eigen_vals))
    pos, neg = float(np.sum(ev[ev > 0])), float(abs(np.sum(ev[ev < 0])))
    return neg / pos if pos > 0 else 0.0


@dataclass
class ITEStepStats:
    bp_iterations: int = 0
    bp_error: float = 0.0
    als_iterations: int = 0
    truncation_distance: float = 0.0
    t_bp: float = 0.0
    t_reduce: float = 0.0
    t_update: float = 0.0
    env_metrics: MatrixMetrics | None = None      # of the RDM after the update (what ite_update_unit_cell returns, :183-205)
    saved_to: str | None = None


def ite_edge_update(unit_cell: UnitCell, messages: dict | None, N: int, mode: str, edge: str, delta_t: float, bp_config: BPConfig,
                    chi: int, h=None, normalize: bool = True, save: bool | str = False):
    """one loop body of ite_per_mode with bp_every_edge=True: -> (unit_cell, messages, energy_after, ITEStepStats).
    ``save``: keep a copy of the updated unit cell on disk as the reference does after every update (_tn_update.py:203);
    True = default folder, a string = that folder.  The write happens on the background saver thread (persistence.py)."""
    st = ITEStepStats()
    h = ite.heisenberg_afm() if h is None else np.asarray(h)
    g = ite.g_from_exp_h(h, delta_t)
    B = backend()
    t0 = time.perf_counter()
    tn = bp.KagomeTNRepeatedUnitCell(unit_cell, N)
    messages, bp_stats = bp.robust_belief_propagation(tn, messages, bp_config)
    st.bp_iterations, st.bp_error = bp_stats.iterations, bp_stats.final_error
    t1 = time.perf_counter()
    env12 = reduce_to_core(unit_cell, messages, N, chi)
    ti, tj, env, info = edge_tn(unit_cell, env12, N, mode, edge, chi)
    t2 = time.perf_counter()
    d_virtual = ti.shape[1]
    aux = {}
    ti_new, tj_new, origin_eigen_vals = ite.apply_2local_gate(B, g, d_virtual, ti, tj, env, aux=aux)
    # _measures_on_edge before and after the update (_tn_update.py:181, 190): both RDMs from the reduced environment the gate
    # application has built anyway (same contraction as rho_ij, two passes over the ring tensors less); a trivial / product
    # gate does not build it
    check_rdms_metrics(aux["rho_before"] if "rho_before" in aux else ite.rho_ij(B, ti, tj, env))
    last = getattr(ite.ALS_optimization, "last", None)
    if last:
        st.als_iterations, st.truncation_distance = last["iterations"], last["distance"]
    rho = aux["rho_after"] if "rho_after" in aux else ite.rho_ij(B, ti_new, tj_new, env)
    energy = float(np.real(np.dot(np.asarray(rho).flatten(), h.flatten())))
    st.env_metrics = check_rdms_metrics(rho)
    st.env_metrics.other["original_negativity_ratio"] = _original_negativity_ratio(origin_eigen_vals)
    if normalize:
        ti_new = B.scale(ti_new, 1.0 / B.norm(ti_new))
        tj_new = B.scale(tj_new, 1.0 / B.norm(tj_new))
    new_cell = edge_env.write_back(unit_cell.tensors(), info, ti_new, tj_new)
    t3 = time.perf_counter()
    st.t_bp, st.t_reduce, st.t_update = t1 - t0, t2 - t1, t3 - t2
    out_cell = UnitCell(*new_cell, unit_cell._file_name if isinstance(unit_cell, UnitCell) else None)
    if save:
        st.saved_to = out_cell.save(folder=save if isinstance(save, str) else None, asynchronous=True)
    return out_cell, messages, energy, st


def ite_per_mode(unit_cell: UnitCell, messages: dict | None, N: int, mode: str, edge_order, bp_config: BPConfig, chi: int, h=None):
    """(main.py:540-594)  edge_order: iterable of (edge, delta_t)  -> (unit_cell, messages, edge_energies, [stats])"""
    energies, stats = {}, []
    for e, dt in edge_order:
        unit_cell, messages, energy, st = ite_edge_update(unit_cell, messages, N, mode, e, dt, bp_config, chi, h)
        energies[f"({e[0]}, {e[1]})"] = energy
        stats.append(st)
    return unit_cell, messages, energies, stats
