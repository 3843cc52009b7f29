"""Simple update on the device (KBP_OP_SU) against the numpy oracle, batch independence, the identity gate, the known D = 2
answer and the ensemble hook.  Only gauge-invariant quantities are compared: the SU(2) multiplets of the Heisenberg model
leave individual singular vectors undetermined."""
import math

import numpy as np
import pytest

from kagomeperiodicbp_b200 import edge_env, ite
from kagomeperiodicbp_b200 import simple_update as su
from kagomeperiodicbp_b200.containers import BPConfig, UnitCell
from oracle import su_np

pytestmark = pytest.mark.gpu

TABLE = su.bond_table()


def _oracle(cell, schedule, tol=0.0):
    D = cell.A.shape[1]
    gammas, lams = list(cell.tensors()), [np.full(D, 1 / math.sqrt(D))] * 6
    for dt, n in schedule:
        gammas, lams, _, _ = su_np.simple_update(gammas, lams, ite.g_from_exp_h(ite.heisenberg_afm(), dt), n, tol, TABLE)
    return gammas, lams


def _lams(r):
    return [r.lambdas[e] for e in edge_env.EDGES]


def _canonical_error(gammas, lams):
    legb = su_np.leg_bonds(TABLE)
    worst = 0.0
    for s, G in enumerate(gammas):
        D = G.shape[1]
        for l in range(4):
            T = np.moveaxis(su_np._with_outer(G, s, l, lams, legb), l + 1, -1).reshape(-1, D)
            R = T.T @ T.conj()
            worst = max(worst, float(np.linalg.norm(R * D / np.trace(R) - np.eye(D))))
    return worst


@pytest.mark.parametrize("D", [2, 3, 4, 6])
@pytest.mark.parametrize("steps, tol", [(1, 1e-12), (50, 1e-9)])
def test_kernel_matches_oracle(D, steps, tol):
    cells = [UnitCell.random(2, D, seed=100 + s) for s in range(5)]
    schedule = ((0.05, steps),)
    res = su.simple_update(cells, schedule=schedule, tol=0.0)
    for cell, r in zip(cells, res):
        assert r.steps == [steps]
        gammas, lams = _oracle(cell, schedule)
        for b, e in enumerate(edge_env.EDGES):
            assert np.max(np.abs(r.lambdas[e] - lams[b])) < tol * np.max(lams[b]), (D, e)
            assert np.max(np.abs(r.rdms[e] - su_np.bond_rdm(gammas, lams, b, TABLE))) < tol, (D, e)
            # the device RDM is that of the device state
            assert np.max(np.abs(r.rdms[e] - su_np.bond_rdm(list(r.gammas), _lams(r), b, TABLE))) < 1e-12


def test_batch_independence():
    cells = [UnitCell.random(2, 2, seed=s) for s in range(8)]
    schedule = ((0.1, 300),)
    batch = su.simple_update(cells, schedule=schedule, tol=1e-5)
    alone = su.simple_update(cells[:1], schedule=schedule, tol=1e-5)[0]
    assert len({r.steps[0] for r in batch}) > 1, [r.steps for r in batch]
    for e in edge_env.EDGES:
        assert np.array_equal(alone.lambdas[e], batch[0].lambdas[e])
        assert np.array_equal(alone.rdms[e], batch[0].rdms[e])
    for a, b in zip(alone.gammas, batch[0].gammas):
        assert np.array_equal(a, b)
    assert alone.steps == batch[0].steps


def test_identity_gate_reaches_the_canonical_gauge():
    cells = [UnitCell.random(2, D, seed=7) for D in (3,)] * 2
    res = su.simple_update(cells, h=np.zeros((2, 2, 2, 2)), schedule=((0.1, 200),), tol=1e-14)
    for r in res:
        assert _canonical_error(list(r.gammas), _lams(r)) < 1e-10


BP_CFG = dict(trunc_dim=8, msg_diff_terminate=1e-6, msg_diff_good_enough=1e-5, damping=0.1, init_msg="UQ", max_iterations=50)


def test_known_answer_D2():
    """SU of a random D = 2 cell, evaluated with block BP at the settings of test_ite_descends_into_the_known_energy_band, lies
    near the variPEPS SU value -0.38620; full-update ITE started there ends in that test's band."""
    from kagomeperiodicbp_b200 import belief_propagation as bp
    from kagomeperiodicbp_b200 import ite_flow
    D, N, chi = 2, 2, 18
    r = su.simple_update([UnitCell.random(2, D, seed=0)])[0]
    assert r.deltas[-1] < 1e-4, r.deltas
    cfg = BPConfig(**BP_CFG)
    cell = r.unit_cell
    msgs, _ = bp.robust_belief_propagation(bp.KagomeTNRepeatedUnitCell(cell, N), None, cfg)
    e_su = ite_flow.measure_energies(cell, msgs, N, chi, mode="A").mean_energy
    assert -0.396 < e_su < -0.376, e_su
    for dt, sweeps in ((0.1, 3), (0.05, 2)):
        for _ in range(sweeps):
            for mode in edge_env.MODES:
                cell, msgs, _, _ = ite_flow.ite_per_mode(cell, msgs, N, mode, [(e, dt) for e in edge_env.EDGES], cfg, chi)
    e_fu = ite_flow.measure_energies(cell, msgs, N, chi, mode="A").mean_energy
    assert -0.4047 < e_fu < -0.375, e_fu


def test_ensemble_su_init():
    from kagomeperiodicbp_b200.ensemble import RESULT_KEYS, run_ensemble
    rows = run_ensemble(seeds=[0, 1], D=2, N=2, init="su")
    assert [r["seed"] for r in rows] == [0, 1]
    for r in rows:
        assert list(r.keys()) == RESULT_KEYS
        assert -0.396 < r["energy"] < -0.376, r
