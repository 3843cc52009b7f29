"""GPU tier: the batched measurement on the device -- the reference's RDMs / energies from its converged messages, the best D = 2
unit cell measured inside a batch of random cells against the reference's edge energies, batched against per-cell
measurements at D = 4, N = 3, independence of a cell's result from its place in the batch, graph replay against the first
host-driven run, and the ensemble launcher's energies."""
import numpy as np
import pytest

from helpers import golden
from test_measure_batch_cpu import assert_same_measurements, check_golden, random_cells_after_bp

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module", autouse=True)
def own_engines():
    """this module's side chains and measurement programs run on engines of its own, closed at the end.  Its batches
    re-reserve engines at other numbers of chains, which drops the captured graphs an engine holds; the process-wide side
    engines keep theirs, and the arenas of the D = 4 batches (8 GB per chain) are freed when the module is done."""
    from kagomeperiodicbp_b200 import belief_propagation as bp
    from kagomeperiodicbp_b200 import ite_flow
    from kagomeperiodicbp_b200.engine import Engine
    engines = {}

    def get(key="default", device=0):
        if (key, device) not in engines:
            engines[(key, device)] = Engine(device)
        return engines[(key, device)]
    saved = bp.get_engine, ite_flow._measure_engine
    bp.get_engine, ite_flow._measure_engine = get, lambda device: get("measure", device)
    yield
    bp.get_engine, ite_flow._measure_engine = saved
    for e in engines.values():
        e.close()


@pytest.mark.parametrize("D", [2, 3])
def test_batched_measurement_matches_reference(D):
    check_golden(D)


@pytest.mark.parametrize("N", [2, 3])
def test_best_unit_cell_inside_a_batch(N):
    """the known answer of test_known_answer_gpu.py, with the best cell in the middle of a batch of random cells."""
    from kagomeperiodicbp_b200 import belief_propagation as bp
    from kagomeperiodicbp_b200 import ensemble, ite_flow
    from kagomeperiodicbp_b200.containers import BPConfig, UnitCell
    g = golden("best_D2.npz")
    chi_bp, chi, iters, term, damping = g[f"N{N}_cfg"].tolist()
    cell = UnitCell(g["A"], g["B"], g["C"])
    cfg = BPConfig(trunc_dim=int(chi_bp), msg_diff_terminate=term, damping=None if damping < 0 else damping, init_msg="UQ")
    tn = bp.KagomeTNRepeatedUnitCell(cell, N)
    tn.connect_uniform_messages()
    msgs, stats = bp.belief_propagation(tn, tn.messages, cfg)
    assert stats.iterations == int(iters)
    others = [UnitCell.random(2, 2, seed=s) for s in (21, 22, 23)]
    rcfg = BPConfig(trunc_dim=int(chi_bp), msg_diff_terminate=1e-8, damping=0.1, init_msg="UQ", max_iterations=30)
    omsgs = [r[0] for r in ensemble.belief_propagation_batch(N, others, rcfg, batch=3)]
    assert all(bp._msg_shapes(m) == bp._msg_shapes(msgs) for m in omsgs)         # one shape group: one launch
    cells, mlist = others[:2] + [cell] + others[2:], omsgs[:2] + [msgs] + omsgs[2:]
    ms = ite_flow.measure_energies_batch(cells, mlist, N, int(chi), g["h"], mode="A", batch=len(cells))
    ref = dict(zip(g[f"N{N}_edges"].tolist(), g[f"N{N}_edge_energies"].tolist()))
    for e, v in ref.items():
        assert abs(ms[2].energies[f"({e[0]}, {e[1]})"] - v) < 1e-8, (e, ms[2].energies, v)
    assert abs(ms[2].mean_energy - float(g["file_energy"][0])) < 3e-4


@pytest.fixture(scope="module")
def d4n3_cells(own_engines):
    D, N = 4, 3
    return random_cells_after_bp(D, N, range(100, 108), batch=8)


def test_d4_n3_batch_equals_single_cell_measurements(d4n3_cells):
    from kagomeperiodicbp_b200 import ite_flow
    cells, msgs = d4n3_cells
    N, chi = 3, 2 * 4 * 4 + 10
    ms = ite_flow.measure_energies_batch(cells, msgs, N, chi, batch=8)
    for cell, m_msgs, m in zip(cells, msgs, ms):
        assert_same_measurements(m, ite_flow.measure_energies(cell, m_msgs, N, chi), 1e-10)


def test_rotated_batch_gives_identical_results(d4n3_cells):
    """a cell's result does not depend on its place in the batch.  Both runs compared are graph launches: a program's first,
    host-driven run at this nb records how many subspace rounds each truncation needed and the captured graph does those
    iterations up front (DESIGN section 3), which at D = 4 changes the last bits -- that is the execution mode, not the
    cell's position, so the warm-up call below takes the host-driven run of every program involved."""
    from kagomeperiodicbp_b200 import ite_flow
    cells, msgs = d4n3_cells
    N, chi = 3, 2 * 4 * 4 + 10
    ite_flow.measure_energies_batch(cells, msgs, N, chi, batch=8)
    eng = ite_flow._measure_engine(0)
    before = eng.graph_counters()
    base = ite_flow.measure_energies_batch(cells, msgs, N, chi, batch=8)
    r = 3
    rot = ite_flow.measure_energies_batch(cells[r:] + cells[:r], msgs[r:] + msgs[:r], N, chi, batch=8)
    after = eng.graph_counters()
    assert after["graph_replays"] >= before["graph_replays"] + 2, (before, after)
    for k, m in enumerate(rot):
        b = base[(k + r) % 8]
        for e in m.rdms:
            assert np.array_equal(m.rdms[e], b.rdms[e]), (k, e)
        assert m.energies == b.energies


def test_graph_replay_equals_first_host_driven_run():
    """a program first runs host-driven, is captured on its second run and replayed from then on: all three bit-identical.
    At D = 2 every truncation of the program is settled in its first subspace round (or by the exact Jacobi path), so the
    graph does the same iterations as the host-driven run."""
    from kagomeperiodicbp_b200 import ite_flow
    D, N, chi = 2, 2, 17                                   # a bond no other test compiles: this program is new here
    cells, msgs = random_cells_after_bp(D, N, (31, 32, 33), batch=3)
    eng = ite_flow._measure_engine(0)
    before = eng.graph_counters()
    runs = [ite_flow.measure_energies_batch(cells, msgs, N, chi, batch=3) for _ in range(3)]
    after = eng.graph_counters()
    assert after["graph_captures"] > before["graph_captures"] and after["graph_replays"] > before["graph_replays"], (before, after)
    for ms in runs[1:]:
        for a, b in zip(runs[0], ms):
            for e in a.rdms:
                assert np.array_equal(a.rdms[e], b.rdms[e]), e


def test_run_ensemble_energies_equal_per_cell_measurement(monkeypatch):
    from kagomeperiodicbp_b200 import ensemble, ite_flow
    seen = []
    batched = ite_flow.measure_energies_batch

    def spy(cells, messages_list, *a, **k):
        seen.append((list(cells), list(messages_list), a))
        return batched(cells, messages_list, *a, **k)
    monkeypatch.setattr(ite_flow, "measure_energies_batch", spy)
    D, N = 2, 2
    rows = ensemble.run_ensemble(range(5), D, N, batch=4)
    (cells, msgs, (n, chi)), = seen
    assert n == N and len(rows) == len(cells) == 5
    for row, cell, m in zip(rows, cells, msgs):
        assert abs(row["energy"] - ite_flow.measure_energies(cell, m, N, chi).mean_energy) < 1e-10, row
