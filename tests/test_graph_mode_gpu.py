"""GPU tier: programs executed as ONE CUDA graph -- the data-dependent loops of the truncated SVD are conditional WHILE / IF
nodes driven by device-side decision kernels -- must give what the host-driven execution of the same program gives, for every
branch: accepted at the first check, further rounds, hand-over to the exact (block-Jacobi) path, the Householder-reduced
path, ensembles whose chains take different branches."""
import numpy as np
import pytest

from kagomeperiodicbp_b200.program import Program
from kagomeperiodicbp_b200.runtime import Compiled

pytestmark = pytest.mark.gpu

rng = np.random.default_rng(4321)


def rnd(*s):
    return rng.normal(size=s) + 1j * rng.normal(size=s)


@pytest.fixture(scope="module")
def engines():
    from kagomeperiodicbp_b200.engine import Engine
    host, graph = Engine(0), Engine(0)
    host.graph_policy(1 << 40, False)          # never captured: host-driven loops
    graph.graph_policy(0, True)                # captured at first sight, whatever the length
    yield host, graph
    host.close()
    graph.close()


def with_spectrum(m, n, s):
    u, _, vh = np.linalg.svd(rnd(m, n), full_matrices=False)
    return (u * s) @ vh


def compile_svd(m, n, keep, n_slots=8):
    p = Program(n_slots)
    t = p.input("i0", (m, n))
    us, vh = p.svd_trunc(t, keep, True, 0, 1)
    return Compiled(p, [("i0", t)], [("o0", us), ("o1", vh)])


def check(a, us, vh, sl, keep, tol=2e-13):
    u, s, v = np.linalg.svd(a, full_matrices=False)
    fro = np.linalg.norm(s)
    ref = (u[:, :keep] * s[:keep]) @ v[:keep]
    gap = max((s[keep - 1] - s[keep]) / s[0], 1e-3) if keep < len(s) else 1.0
    assert np.linalg.norm(us @ vh * fro - ref) <= tol * fro / gap
    terr = np.sqrt(np.sum(s[keep:] ** 2) / np.sum(s ** 2))
    assert abs(sl[1] - terr) <= 1e-10
    assert abs(sl[0] - np.log(fro)) <= 1e-12 * max(1, abs(np.log(fro)))
    assert sl[-1] == 0


CASES = {
    # name: (m, n, keep, spectrum builder)
    "first_check": (512, 512, 32, lambda p: np.sort(np.exp(-0.1 * np.arange(p)) * (1 + 0.3 * rng.random(p)))[::-1]),
    "more_rounds": (512, 512, 32, lambda p: np.exp(-0.02 * np.arange(p))),
    "collapse_exact": (256, 256, 32, lambda p: np.where(np.arange(p) < 20, 1.0, np.where(np.arange(p) < 60, 1e-9, 0.0))),
    # kept spectrum over more than six decades, but the block resolves a direction below the kept ones: stays on the subspace path
    "collapse_resolved": (512, 512, 32, lambda p: np.exp(-0.45 * np.arange(p))),
    "reduced_wide": (64, 512, 32, lambda p: np.exp(-0.15 * np.arange(p))),
    "reduced_tall": (512, 64, 32, lambda p: np.exp(-0.15 * np.arange(p))),
    "plain_exact": (200, 160, 150, lambda p: np.exp(-0.05 * np.arange(p))),
    "d3_size": (162, 162, 18, lambda p: np.exp(-0.15 * np.arange(p))),
}


@pytest.mark.parametrize("name", list(CASES))
def test_graph_equals_host_driven(engines, name):
    host, graph = engines
    m, n, keep, spec = CASES[name]
    a = with_spectrum(m, n, spec(min(m, n))) * 2.5
    comp = compile_svd(m, n, keep)
    c0 = graph.svd_counters()
    oh, sh, _ = comp.run(host, [{"i0": a}])
    res = [comp.run(graph, [{"i0": a}]) for _ in range(3)]             # capture + 2 replays
    c1 = graph.svd_counters()
    assert c1["graph_replays"] - c0["graph_replays"] == 3 and c1["graph_capture_failures"] == c0["graph_capture_failures"], (c0, c1)
    for og, sg, _ in res:
        # same kernels, same order, same decisions: bitwise equal
        assert np.array_equal(og[0]["o0"], oh[0]["o0"]) and np.array_equal(og[0]["o1"], oh[0]["o1"]), name
        assert np.array_equal(sg, sh)
    if name != "collapse_exact":
        check(a, oh[0]["o0"], oh[0]["o1"], sh[0], keep)
    else:
        us, vh = oh[0]["o0"], oh[0]["o1"]
        assert np.linalg.norm(us @ vh * np.linalg.norm(a) - a) <= 1e-8 * np.linalg.norm(a)     # rank 60 > keep, tail 1e-9
        assert sh[0, -1] == 0
    d = {k: c1[k] - c0[k] for k in c1}
    if name == "first_check":
        assert d["subspace"] == 3 and d["subspace_iterations"] == 3 * 7 and d["subspace_fallback"] == 0, d
    if name == "more_rounds":
        assert d["subspace"] == 3 and d["subspace_iterations"] > 3 * 7, d
    if name == "collapse_exact":
        assert d["subspace_fallback"] == 3 and d["block_jacobi"] == 3 and d["block_jacobi_sweeps"] >= 3, d
    if name == "collapse_resolved":
        assert d["subspace"] == 3 and d["subspace_fallback"] == 0 and d["block_jacobi"] == 0, d
    if name.startswith("reduced"):
        assert d["reduced"] == 3 and d["block_jacobi"] == 0, d
    if name == "plain_exact":
        assert d["block_jacobi"] == 3, d


def test_graph_ensemble_chains_take_different_branches(engines):
    """four chains in one launch: accepted at once / needs more rounds / exact path / accepted -- each must get its own result."""
    host, graph = engines
    m = n = 256
    keep = 32
    p = np.arange(m)
    specs = [np.exp(-0.1 * p), np.exp(-0.02 * p), np.where(p < 20, 1.0, np.where(p < 60, 1e-9, 0.0)), np.exp(-0.2 * p)]
    mats = [with_spectrum(m, n, s) * (1.0 + c) for c, s in enumerate(specs)]
    comp = compile_svd(m, n, keep)
    batch = [{"i0": a} for a in mats]
    oh, sh, _ = comp.run(host, batch)
    c0 = graph.svd_counters()
    for _ in range(2):
        og, sg, _ = comp.run(graph, batch)
        for c in range(4):
            assert np.array_equal(og[c]["o0"], oh[c]["o0"]) and np.array_equal(og[c]["o1"], oh[c]["o1"]), c
        assert np.array_equal(sg, sh)
    c1 = graph.svd_counters()
    d = {k: c1[k] - c0[k] for k in c1}
    assert d["subspace"] == 6 and d["subspace_fallback"] == 2 and d["block_jacobi"] == 2, d
    for c in (0, 1, 3):
        check(mats[c], oh[c]["o0"], oh[c]["o1"], sh[c], keep)
    # each chain alone gives the same truncated state as inside the ensemble (chains do not influence each other; the GEMM
    # tiling depends on the number of chains, so only to rounding)
    for c in range(4):
        o1, s1, _ = comp.run(host, [batch[c]])
        assert np.linalg.norm(o1[0]["o0"] @ o1[0]["o1"] - oh[c]["o0"] @ oh[c]["o1"]) <= 1e-9, c
        assert np.allclose(s1[0], sh[c], atol=1e-10)


def test_whole_side_program_as_graph():
    """a D=3, N=2 block side program (chain + normalisation + overlap + damping, 160 x 162 subspace truncations) run as a graph
    equals its host-driven run bitwise; replays launch nothing from the host but the graph."""
    from kagomeperiodicbp_b200 import belief_propagation as bp
    from kagomeperiodicbp_b200.containers import BPConfig, UnitCell
    from kagomeperiodicbp_b200.engine import Engine
    D, N = 3, 2
    cell = UnitCell.random(2, D, seed=3)
    cfg = BPConfig(trunc_dim=2 * D * D, msg_diff_terminate=1e-6, damping=0.1, init_msg="UQ")
    msgs = bp.initial_messages(D, N, "UQ")
    for _ in range(2):
        msgs = bp.bp_step_batch(N, [cell], [msgs], cfg)[0][1]
    comp = bp.compile_side_program(N, 2, D, "D", 2 * D * D, bp._msg_shapes(msgs), 0.1)
    batch = [bp._side_inputs(cell, msgs, comp)]
    host, graph = Engine(0), Engine(0)
    try:
        host.graph_policy(1 << 40, False)
        oh, sh, rh = comp.run(host, batch)
        assert not graph.graph_ready(comp.words)
        o1, s1, _ = comp.run(graph, batch)               # first sight: host-driven
        assert graph.graph_ready(comp.words)
        o2, s2, _ = comp.run(graph, batch)               # captured
        o3, s3, _ = comp.run(graph, batch)               # replayed
        gc = graph.graph_counters()
        assert gc["graph_captures"] == 1 and gc["graph_replays"] == 2 and gc["graph_capture_failures"] == 0, gc
        for o, s in ((o1, s1), (o2, s2), (o3, s3)):
            for k in oh[0]:
                assert np.array_equal(o[0][k], oh[0][k]), k
            assert np.array_equal(s, sh)
    finally:
        host.close()
        graph.close()

