"""Simple update without a GPU: the bond table, the numpy oracle against dense linear algebra, and the host side of the
batched program (packing, the op words, unpacking) on the numpy interpreter with the oracle standing in for the kernel."""
import math
import struct

import numpy as np
import pytest

from kagomeperiodicbp_b200 import edge_env, ite
from kagomeperiodicbp_b200 import simple_update as su
from kagomeperiodicbp_b200.containers import UnitCell
from kagomeperiodicbp_b200.engine import OP_SU
from kagomeperiodicbp_b200.lattice import LATTICE_OPPOSITE, SITE_DIRS, SITE_KINDS
from oracle import su_np
from np_vm import NumpyEngine

TABLE = su.bond_table()
IDENTITY = np.einsum("ab,cd->abcd", np.eye(2), np.eye(2)).astype(np.complex128)


def random_state(D, seed):
    rs = np.random.RandomState(seed)
    gammas = list(UnitCell.random(2, D, seed=seed).tensors())
    lams = [np.sort(rs.rand(D) + 0.05)[::-1] for _ in range(6)]
    return gammas, [l / np.linalg.norm(l) for l in lams]


def canonical_error(gammas, lams):
    """max over sites and legs of | sum Gamma lambda^2_others Gamma^* / (tr / D) - 1 |"""
    legb = su_np.leg_bonds(TABLE)
    worst = 0.0
    for s, G in enumerate(gammas):
        D = G.shape[1]
        for l in range(4):
            T = np.moveaxis(su_np._with_outer(G, s, l, lams, legb), l + 1, -1).reshape(-1, D)
            R = T.T @ T.conj()
            worst = max(worst, float(np.linalg.norm(R * D / np.trace(R) - np.eye(D))))
    return worst


def test_bond_table_pairs_every_leg_once_in_opposite_directions():
    seen = []
    for i, li, j, lj in TABLE:
        seen += [(i, li), (j, lj)]
        assert i != j
        di, dj = SITE_DIRS[SITE_KINDS[i]][li], SITE_DIRS[SITE_KINDS[j]][lj]
        assert LATTICE_OPPOSITE[di] == dj, (i, li, j, lj)
    assert sorted(seen) == [(s, l) for s in range(3) for l in range(4)]
    assert len(TABLE) == len(edge_env.EDGES) == 6


@pytest.mark.parametrize("D", [2, 3])
def test_oracle_bond_update_is_the_best_rank_D_approximation(D):
    gammas, lams = random_state(D, seed=D)
    g = ite.g_from_exp_h(ite.heisenberg_afm(), 0.3)
    for b in range(6):
        psi = su_np.bond_contraction(gammas, lams, b, TABLE)                 # [(p, outer_i), (q, outer_j)]
        n = psi.shape[0] // 2
        dense = np.einsum("PpQq,paqb->PaQb", g, psi.reshape(2, n, 2, n)).reshape(2 * n, 2 * n)
        U, S, Vh = np.linalg.svd(dense)
        best = (U[:, :D] * S[:D]) @ Vh[:D]
        g2, l2 = su_np.bond_update(gammas, lams, b, g, TABLE)
        new = su_np.bond_contraction(g2, l2, b, TABLE)
        ph = np.vdot(new, best) / abs(np.vdot(new, best))
        err = np.linalg.norm(best / np.linalg.norm(best) - ph * new / np.linalg.norm(new))
        assert err < 1e-12, (D, b, err)
        assert abs(np.linalg.norm(l2[b]) - 1) < 1e-14 and np.all(np.diff(l2[b]) <= 0)
        gammas, lams = g2, l2


@pytest.mark.parametrize("D", [2, 3])
def test_identity_gate_keeps_the_bond_and_reaches_the_canonical_gauge(D):
    gammas, lams = random_state(D, seed=10 + D)
    for b in range(6):
        before = su_np.bond_contraction(gammas, lams, b, TABLE)
        g2, l2 = su_np.bond_update(gammas, lams, b, IDENTITY, TABLE)
        after = su_np.bond_contraction(g2, l2, b, TABLE)
        ph = np.vdot(after, before) / abs(np.vdot(after, before))
        assert np.linalg.norm(before / np.linalg.norm(before) - ph * after / np.linalg.norm(after)) < 1e-13
    assert canonical_error(gammas, lams) > 1e-2
    gammas, lams, steps, delta = su_np.simple_update(gammas, lams, IDENTITY, 200, 1e-14, TABLE)
    assert canonical_error(gammas, lams) < 1e-10, (steps, delta)


# ---- the batched program on the numpy interpreter --------------------------------------------------------------------------
SU_WORDS = 38


def _op_len(w, i):
    from kagomeperiodicbp_b200.engine import OP_PERMUTE
    assert w[i] == OP_PERMUTE, "an SU program holds copies and SU ops only"
    return 5 + 2 * w[i + 4]


class OracleSUEngine(NumpyEngine):
    """the numpy interpreter with KBP_OP_SU executed by the oracle"""

    def _run_chain(self, w, ar, sl):
        i = 0
        while i < len(w):
            if w[i] != OP_SU:
                k = _op_len(w, i)
                super()._run_chain(w[i:i + k], ar, sl)
                i += k
                continue
            v = w[i + 1:i + SU_WORDS]
            d, D, steps = v[6], v[7], v[8]
            (tol,) = struct.unpack("d", struct.pack("q", v[9]))
            bonds = [tuple(v[13 + 4 * b:17 + 4 * b]) for b in range(6)]
            n = d * D ** 4
            gammas = [ar[v[s]:v[s] + n].reshape(d, D, D, D, D).copy() for s in range(3)]
            lams = list(np.real(ar[v[3]:v[3] + 6 * D]).reshape(6, D))
            gate = ar[v[4]:v[4] + d ** 4].reshape(d, d, d, d)
            gammas, lams, done, delta = su_np.simple_update(gammas, lams, gate, steps, tol, bonds)
            for s in range(3):
                ar[v[s]:v[s] + n] = gammas[s].ravel()
            ar[v[3]:v[3] + 6 * D] = np.concatenate(lams)
            ar[v[5]:v[5] + 6 * d ** 4] = np.concatenate([su_np.bond_rdm(gammas, lams, b, bonds).ravel() for b in range(6)])
            sl[v[10]], sl[v[11]], sl[v[12]] = done, delta, 0
            self._launches += 1
            i += SU_WORDS


def test_program_packing_matches_the_oracle():
    D = 2
    cells = [UnitCell.random(2, D, seed=s) for s in (3, 4, 5)]
    schedule = ((0.1, 3), (0.05, 2))
    res = su.simple_update(cells, schedule=schedule, tol=0.0, engine=OracleSUEngine())
    h = ite.heisenberg_afm()
    for cell, r in zip(cells, res):
        gammas, lams = list(cell.tensors()), [np.full(D, 1 / math.sqrt(D))] * 6
        for dt, n in schedule:
            gammas, lams, steps, _ = su_np.simple_update(gammas, lams, ite.g_from_exp_h(h, dt), n, 0.0, TABLE)
        assert r.steps == [3, 2] and r.converged == [False, False]
        for b, e in enumerate(edge_env.EDGES):
            assert np.allclose(r.lambdas[e], lams[b], rtol=0, atol=1e-13)
            rho = su_np.bond_rdm(gammas, lams, b, TABLE)
            assert np.allclose(r.rdms[e], rho, rtol=0, atol=1e-13)
            assert abs(r.energies[f"({e[0]}, {e[1]})"] - np.real(np.dot(rho.ravel(), h.ravel()))) < 1e-13
        assert abs(r.energy_per_site - sum(r.energies.values()) / 3) < 1e-15
        for s, T in enumerate(su_np.to_unit_cell_tensors(gammas, lams, TABLE)):
            assert np.allclose(r.unit_cell.tensors()[s], T, rtol=0, atol=1e-13)


class _NoEngine:
    def __getattr__(self, name):
        raise AssertionError(f"engine used: {name}")


@pytest.mark.parametrize("d, D", [(2, 7), (3, 2), (2, 1)])
def test_unsupported_dimensions_are_rejected_before_launch(d, D):
    with pytest.raises(ValueError):
        su.simple_update([UnitCell.random(d, D, seed=0)], engine=_NoEngine())
