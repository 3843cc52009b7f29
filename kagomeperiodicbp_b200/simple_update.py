"""Simple-update (SU) initial states on the device: the Kagome simple update of Jiang, Weng and Xiang (PRL 101, 090603 (2008))
on the Gamma / lambda representation of the three-site unit cell, for a batch of cells in one launch per schedule stage (one
CTA per cell, KBP_OP_SU, csrc/k_su.cu).  The resulting cell (sqrt(lambda) absorbed on both ends of every bond) is the usual
starting point of full-update ITE; the SU-environment energy is the quick estimate that comes with it.

The six bonds of the unit cell and the Trotter order (one SU step = the six bond updates in ``bond_table()`` order, first
order) are decided here and passed to the kernel as op arguments.
"""
from __future__ import annotations

import functools
from dataclasses import dataclass, field

import numpy as np

from . import edge_env, ite
from .containers import UnitCell
from .engine import BubbleConError
from .lattice import SITE_KINDS, get_block
from .program import Program
from .runtime import Compiled, get_engine

SITES = "ABC"
DEFAULT_SCHEDULE = ((0.1, 500), (0.05, 500), (0.01, 1000))


@functools.lru_cache(maxsize=None)
def bond_table() -> tuple:
    """the six bonds (site_i, leg_i, site_j, leg_j) of the unit cell (sites 0, 1, 2 = A, B, C; virtual legs 0..3 in UnitCell
    order), one per ITE edge in ``edge_env.EDGES`` order and oriented as that edge's EdgeTN in mode A (site_i = T_i), so the SU
    RDMs have the site order of ``ite_flow.measure_energies``'.  Three bonds lie inside the upper triangle, three join it to
    neighbouring triangles.  The legs are read off the size-2 block of ``lattice``: the edge's two sites are the central
    triangle's sites or their neighbours, and each leg is where the shared edge label sits."""
    blk = get_block(2)
    edges = edge_env.tables()["modes"]["A"]["edges"]

    def site_index(node):
        bulk = [set(e.split("-")) for e in node["edges"] if all(x.isdigit() for x in e.split("-"))]
        return int(set.intersection(*bulk).pop())

    out = []
    for name in edge_env.EDGES:
        ends = []
        nodes = edges[name]["nodes"][:2]
        shared = (set(nodes[0]["edges"]) & set(nodes[1]["edges"])).pop()
        for node in nodes:
            s = blk.sites[site_index(node)]
            assert SITES[SITE_KINDS.index(s.kind)] == node["name"]
            ends += [SITE_KINDS.index(s.kind), s.edges.index(shared)]
        out.append(tuple(ends))
    return tuple(out)


def leg_bonds() -> list:
    """legb[site][leg] = index of the bond (in ``bond_table()``) the virtual leg belongs to."""
    legb = [[None] * 4 for _ in range(3)]
    for b, (i, li, j, lj) in enumerate(bond_table()):
        legb[i][li] = b
        legb[j][lj] = b
    return legb


def check_dimensions(d: int, D: int):
    if d != 2 or not 2 <= D <= 6:
        raise ValueError(f"simple update supports physical dimension 2 and bond dimension 2..6, got d={d}, D={D}")


@dataclass
class SUResult:
    unit_cell: UnitCell                       # sqrt(lambda) absorbed on every virtual leg
    gammas: tuple                             # Gamma_A, Gamma_B, Gamma_C [d, D, D, D, D]
    lambdas: dict                             # edge name -> lambda [D] (unit norm, descending)
    steps: list                               # per schedule stage: SU steps done
    converged: list                           # per schedule stage: last step delta < tol
    deltas: list                              # per schedule stage: last step delta
    rdms: dict = field(default_factory=dict)  # edge name -> two-site RDM [i, i*, j, j*] in the SU environment
    energies: dict = field(default_factory=dict)
    energy_per_site: float = 0.0


def unit_cell_from_gammas(gammas, lambdas) -> UnitCell:
    """A, B, C with sqrt(lambda) of its bond absorbed on every virtual leg (``lambdas`` indexed like ``bond_table()``)."""
    legb = leg_bonds()
    out = []
    for s, G in enumerate(gammas):
        T = np.asarray(G, dtype=np.complex128)
        for l in range(4):
            shape = [1] * 5
            shape[l + 1] = T.shape[l + 1]
            T = T * np.sqrt(np.real(np.asarray(lambdas[legb[s][l]]))).reshape(shape)
        out.append(T)
    return UnitCell(*out)


@functools.lru_cache(maxsize=32)
def _compiled(d: int, D: int, schedule: tuple, tol: float, h_key: bytes) -> Compiled:
    h = np.frombuffer(h_key, dtype=np.complex128).reshape(d, d, d, d)
    prog = Program(n_slots=3 * len(schedule) + 1)           # 3 per stage + the engine's status slot
    ins = [prog.input(s, (d, D, D, D, D)) for s in SITES] + [prog.input("lam", (6, D))]
    # work on copies: a program leaves its inputs as they were uploaded
    gammas = [prog.copy(x) for x in ins[:3]]
    lam = prog.copy(ins[3])
    rdm = prog.new((6, d, d, d, d))
    for k, (dt, steps) in enumerate(schedule):
        gate = prog.const(ite.g_from_exp_h(h, dt))
        prog.simple_update_(gammas, lam, gate, rdm, steps, tol, (3 * k, 3 * k + 1, 3 * k + 2), bond_table())
    outs = list(zip(SITES, gammas)) + [("lam", lam), ("rdm", rdm)]
    return Compiled(prog, list(zip(list(SITES) + ["lam"], ins)), outs, meta={"d": d, "D": D, "schedule": schedule})


def simple_update(cells, h=None, schedule=DEFAULT_SCHEDULE, tol: float = 1e-9, device: int = 0, engine=None) -> list:
    """simple update of every unit cell of ``cells`` (all with the same d, D) in one batched device program, one launch per
    schedule stage ``(dt, max_steps)``; a cell leaves a stage when the largest change of a bond's lambda over one step drops
    below ``tol``.  lambda starts at ones / sqrt(D), Gamma at the cell's tensors.  ``h``: two-site Hamiltonian
    h[i, i*, j, j*] (default: Heisenberg AFM).  ``engine``: an Engine-like object to run on (default: the process's "su"
    engine on ``device``).  -> [SUResult] in input order."""
    cells = list(cells)
    if not cells:
        return []
    d, D = cells[0].A.shape[0], cells[0].A.shape[1]
    check_dimensions(d, D)
    for c in cells:
        for T in c.tensors():
            if np.shape(T) != (d, D, D, D, D):
                raise ValueError(f"every site tensor must be [{d}, {D}, {D}, {D}, {D}], got {np.shape(T)}")
    schedule = tuple((float(dt), int(n)) for dt, n in schedule)
    if not schedule or any(n < 1 for _, n in schedule):
        raise ValueError("the schedule needs at least one stage of at least one step")
    h = ite.heisenberg_afm() if h is None else np.asarray(h, dtype=np.complex128)
    if h.shape != (d, d, d, d):
        raise ValueError(f"h must be [{d}, {d}, {d}, {d}], got {h.shape}")
    comp = _compiled(d, D, schedule, float(tol), np.ascontiguousarray(h).tobytes())
    eng = engine if engine is not None else get_engine("su", device)
    lam0 = np.full((6, D), 1.0 / np.sqrt(D))
    batch = [{"A": c.A, "B": c.B, "C": c.C, "lam": lam0} for c in cells]
    outs, slots, _ = comp.run(eng, batch)
    nst = len(schedule)
    bad = slots[:, [3 * k + 2 for k in range(nst)]].sum(axis=1)
    if np.any(bad > 0):
        raise BubbleConError(f"simple update produced non-finite values in cell(s) {np.nonzero(bad > 0)[0].tolist()}")
    results = []
    for c, o in enumerate(outs):
        lams = np.real(o["lam"])
        gammas = (o["A"], o["B"], o["C"])
        rdms = {e: o["rdm"][b] for b, e in enumerate(edge_env.EDGES)}
        energies = {f"({e[0]}, {e[1]})": float(np.real(np.dot(rdms[e].flatten(), h.flatten()))) for e in edge_env.EDGES}
        deltas = [float(slots[c, 3 * k + 1]) for k in range(nst)]
        results.append(SUResult(unit_cell=unit_cell_from_gammas(gammas, lams), gammas=gammas,
                                lambdas={e: lams[b] for b, e in enumerate(edge_env.EDGES)},
                                steps=[int(slots[c, 3 * k]) for k in range(nst)], converged=[x < tol for x in deltas], deltas=deltas,
                                rdms=rdms, energies=energies, energy_per_site=sum(energies.values()) / 3))
    return results
