"""CPU tier: the batched measurement (two ToCore chains + one compiled core -> edge -> RDM program per batch of cells) on the
op-stream interpreter -- against the reference's RDMs and energies from its converged messages (tests/golden/ite_D2_N2.npz),
against the per-cell ``measure_energies`` on random cells, the shape-only compile at D = 4, N = 3, and the input checks."""
import numpy as np
import pytest

from helpers import golden


@pytest.fixture
def all_vm(vm_engines, monkeypatch):
    from np_vm import NumpyEngine
    import kagomeperiodicbp_b200.linalg as linalg
    from kagomeperiodicbp_b200 import ite_flow
    engines = {}
    monkeypatch.setattr(linalg, "get_engine", lambda key="default", device=0: engines.setdefault(key, NumpyEngine()))
    monkeypatch.setattr(ite_flow, "_backend", linalg.ResidentBackend("vm-ite", arena_elems=1 << 23))
    return engines


def golden_cell_and_messages(D):
    from test_ite_flow_gpu import device_messages
    from kagomeperiodicbp_b200.containers import UnitCell
    g = golden(f"ite_D{D}_N2.npz")
    return g, UnitCell(g["A"], g["B"], g["C"]), device_messages(g, 2)


def check_golden(D, modes=("A", "B", "C")):
    """every mode (direction U) and directions DL / DR (mode A) of the batched measurement against the reference."""
    from kagomeperiodicbp_b200 import edge_env, ite_flow
    g, cell, msgs = golden_cell_and_messages(D)
    chi = int(g["chi"])
    cases = [(mode, "U", f"{mode}_") for mode in modes] + [("A", dr, f"{dr}_A_") for dr in ("DL", "DR")]
    for mode, direction, pre in cases:
        # the golden cell twice in one batch: both chains give the reference's numbers
        ms = ite_flow.measure_energies_batch([cell, cell], [msgs, msgs], 2, chi, g["h"], mode=mode, direction=direction, batch=2)
        for m in ms:
            for e in edge_env.EDGES:
                assert np.max(np.abs(m.rdms[e] - g[f"rdm_{pre}{e}"])) < 1e-9, (D, mode, direction, e)
                assert abs(m.energies[f"({e[0]}, {e[1]})"] - g[f"energy_{pre}{e}"][0]) < 1e-8, (D, mode, direction, e)


def test_batched_measurement_matches_reference_on_the_interpreter(all_vm):
    check_golden(2)


def random_cells_after_bp(D, N, seeds, batch):
    from kagomeperiodicbp_b200 import ensemble
    from kagomeperiodicbp_b200.containers import BPConfig, UnitCell
    cells = [UnitCell.random(2, D, seed=s) for s in seeds]
    cfg = BPConfig(trunc_dim=2 * D * D, msg_diff_terminate=1e-6, damping=0.1, init_msg="UQ", max_iterations=50)
    res = ensemble.belief_propagation_batch(N, cells, cfg, batch=batch)
    return cells, [r[0] for r in res]


def assert_same_measurements(a, b, tol):
    assert a.energies.keys() == b.energies.keys()
    for k in a.energies:
        assert abs(a.energies[k] - b.energies[k]) < tol, k
        assert abs(a.entanglement[k] - b.entanglement[k]) < tol, k
    for e in a.rdms:
        assert np.max(np.abs(np.asarray(a.rdms[e]) - np.asarray(b.rdms[e]))) < tol, e
    for f in "ABC":
        for k in "xyz":
            assert abs(a.expectations[f][k] - b.expectations[f][k]) < tol, (f, k)


def test_batched_measurement_equals_per_cell_measurement(all_vm):
    from kagomeperiodicbp_b200 import ite_flow
    D, N, chi = 2, 2, 18
    cells, msgs = random_cells_after_bp(D, N, (3, 4, 5), batch=2)
    ms = ite_flow.measure_energies_batch(cells, msgs, N, chi, batch=2)
    for cell, m_msgs, m in zip(cells, msgs, ms):
        assert_same_measurements(m, ite_flow.measure_energies(cell, m_msgs, N, chi), 1e-12)


def test_measurement_program_compiles_without_an_engine():
    """D = 4, N = 3: shapes only -- no engine, no device, no host value of any tensor."""
    from kagomeperiodicbp_b200 import belief_propagation as bp
    from kagomeperiodicbp_b200 import edge_env, ite_flow
    D, N, chi = 4, 3, 2 * 4 * 4 + 10
    msg_shapes = bp._msg_shapes(bp.initial_messages(D, N, "UQ"))
    msg_shapes = tuple(tuple((min(a, 2 * D * D), b, min(c, 2 * D * D)) for a, b, c in side) for side in msg_shapes)
    tocore = []
    for side in edge_env.CORE_DIRECTIONS["U"][:2]:
        comp = bp.compile_side_program(N, 2, D, side, chi, msg_shapes, None, depth="ToCore", epilogue=False)
        tocore.append([shape for _, _, shape in comp.out_layout])
    comp = ite_flow.compile_measurement(N, 2, D, chi, "A", "U", tocore)
    assert [name for name, _, _ in comp.out_layout] == [f"rho{k}" for k in range(6)]
    assert all(shape == (2, 2, 2, 2) for _, _, shape in comp.out_layout)
    assert [name for name, _, _ in comp.in_layout][:3] == ["cellA", "cellB", "cellC"]
    assert comp.arena_elems > 0 and len(comp.words) > 0
    assert ite_flow.compile_measurement(N, 2, D, chi, "A", "U", tocore) is comp


def test_traced_tensors_have_no_host_value():
    from kagomeperiodicbp_b200.linalg import TArr, TraceBackend
    from kagomeperiodicbp_b200.program import Program
    p = Program(8)
    B = TraceBackend(p)
    x = TArr(p.input("x", (2, 3)))
    y = B.tensordot(x, x, ([0], [0]), conj_b=True)
    assert y.shape == (3, 3) and B.reshape(y, (-1,)).shape == (9,)
    with pytest.raises(TypeError):
        np.asarray(y)
    with pytest.raises(TypeError):
        y[0]
    with pytest.raises(TypeError):
        B.tensordot(x, np.ones((2, 3)), ([0], [0]))


@pytest.fixture
def no_launch(monkeypatch):
    """any launch fails the test: the input checks must come first."""
    from kagomeperiodicbp_b200 import belief_propagation as bp
    from kagomeperiodicbp_b200 import ite_flow

    def boom(*a, **k):
        raise AssertionError("launched")
    monkeypatch.setattr(bp, "_run_side", boom)
    monkeypatch.setattr(ite_flow, "_measure_engine", boom)


def test_input_errors_raise_before_any_launch(no_launch):
    from kagomeperiodicbp_b200 import belief_propagation as bp
    from kagomeperiodicbp_b200 import ite_flow
    from kagomeperiodicbp_b200.containers import LatticeTensors, UnitCell
    c2, c3 = UnitCell.random(2, 2, seed=0), UnitCell.random(2, 3, seed=0)
    m2, m3 = bp.initial_messages(2, 2, "UQ"), bp.initial_messages(3, 2, "UQ")
    assert ite_flow.measure_energies_batch([], [], 2, 18) == []
    bad = [
        dict(cells=[c2, c3], messages_list=[m2, m3]),                                  # mixed D
        dict(cells=[c2, UnitCell.random(3, 2, seed=1)], messages_list=[m2, m2]),        # mixed d
        dict(cells=[c2, LatticeTensors([c2.A] * 12)], messages_list=[m2, m2]),          # non-repeated block
        dict(cells=[c2], messages_list=[m2], mode="D"),
        dict(cells=[c2], messages_list=[m2], direction="UR"),
        dict(cells=[c2, c2], messages_list=[m2]),
    ]
    for kw in bad:
        args = dict(N=2, chi=18)
        args.update(kw)
        with pytest.raises(ValueError):
            ite_flow.measure_energies_batch(**args)
