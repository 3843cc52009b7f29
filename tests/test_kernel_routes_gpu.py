"""GPU tier: every ZGEMM tile kernel and every truncated-SVD route, each reached by a shape the dispatch mirror
(tests/kernel_routes.py) says reaches it, against exact, extended-precision and gap-free float64 references.

Each SVD case also asserts the route it took from Engine.svd_counters(), so a kernel that breaks and silently hands its
chains to the exact path fails here.  Operands sit between NaN-filled neighbours: a copy or a store that ignores a bound
shows up as a NaN or as a changed canary.  The engine runs programs host-driven (one plain launch per kernel) except in
the split-K test, which compares host-driven, captured and replayed runs of the same program."""
import numpy as np
import pytest

import kernel_routes as kr
from kagomeperiodicbp_b200.program import Program
from kagomeperiodicbp_b200.runtime import Compiled

pytestmark = pytest.mark.gpu

PAD = 8                              # elements of every NaN neighbour (one allocation unit)
CANARY = 1234.5 - 678.25j
NAN = complex(np.nan, np.nan)
S200 = 2.0 ** 200


@pytest.fixture(scope="module")
def eng():
    from kagomeperiodicbp_b200.engine import Engine
    e = Engine(0)
    e.graph_policy(1 << 40, False)   # host-driven: one plain launch per kernel, counters per run
    yield e
    e.close()


def compile_program(inputs, build, n_slots=8):
    """inputs: [(name, shape)] declared in order (so the arena holds them back to back); build(p, {name: DT}) -> outputs"""
    p = Program(n_slots)
    dts = [(nm, p.input(nm, sh)) for nm, sh in inputs]
    outs = build(p, dict(dts))
    return Compiled(p, dts, [(f"o{k}", t) for k, t in enumerate(outs)]), len(outs)


def run(eng, prog, batch):
    comp, nout = prog
    o, sl, rc = comp.run(eng, batch)
    assert rc == 0, rc
    return [[oc[f"o{k}"] for k in range(nout)] for oc in o], sl


# ================================================================================================================ ZGEMM
PAIRS = [(oa, ob) for oa in range(4) for ob in range(4)]
HOMOG = [(0, 0), (1, 2), (2, 3), (3, 1)]          # pairs also run with 2^200 A


def gemm_program(m, n, k):
    ins = [(f"A{o}", kr.stored_operand(np.zeros((m, k)), o).shape) for o in range(4)]
    ins += [(f"S{o}", kr.stored_operand(np.zeros((m, k)), o).shape) for o, _ in HOMOG]
    ins += [(f"B{o}", kr.stored_operand(np.zeros((k, n)), o).shape) for o in range(4)]

    def build(p, t):
        out = [p.matmul(t[f"A{oa}"], t[f"B{ob}"], m, n, k, oa, ob) for oa, ob in PAIRS]
        return out + [p.matmul(t[f"S{oa}"], t[f"B{ob}"], m, n, k, oa, ob) for oa, ob in HOMOG]
    return compile_program(ins, build)


def gemm_inputs(a, b):
    d = {f"A{o}": kr.stored_operand(a, o) for o in range(4)}
    d.update({f"S{o}": kr.stored_operand(a * S200, o) for o, _ in HOMOG})
    d.update({f"B{o}": kr.stored_operand(b, o) for o in range(4)})
    return d


def one_hot_case(rng, pattern, m, n, k):
    """0 dense; 1 one nonzero of A in its last row and last k index; 2 one nonzero of B in the last k index and last column;
    3 one nonzero each, at the last row of A and the last column of B (k index 0)"""
    a, b = kr.int_complex(rng, (m, k)), kr.int_complex(rng, (k, n))
    if pattern == 1:
        v = a[m - 1, k - 1]
        a[:] = 0
        a[m - 1, k - 1] = v if v != 0 else 3 - 5j
    elif pattern == 2:
        v = b[k - 1, n - 1]
        b[:] = 0
        b[k - 1, n - 1] = v if v != 0 else -7 + 2j
    elif pattern == 3:
        a[:] = 0
        b[:] = 0
        a[m - 1, 0], b[0, n - 1] = 8 - 8j, -8 + 7j
    return a, b


def check_homogeneity(res, what):
    for j, pair in enumerate(HOMOG):
        c, h = res[PAIRS.index(pair)], res[len(PAIRS) + j]
        assert np.array_equal(h, c * S200), f"{what}: gemm(2^200 A, B) != 2^200 gemm(A, B) for ops {pair}"


@pytest.mark.parametrize("name", list(kr.GEMM_CASES))
def test_zgemm_route(eng, name):
    """exact (integer data, bitwise), one-hot edges, extended-precision accuracy, 2^200 homogeneity, chain rotation"""
    m, n, k, nb = kr.GEMM_CASES[name]
    r = kr.gemm_route(m, n, k, nb)
    assert (r["tile"], r["fused"], r["rows_on_x"]) == kr.GEMM_EXPECT[name], r
    rng = np.random.default_rng(sum(map(ord, name)))
    prog = gemm_program(m, n, k)
    # exact: every chain of a run gets its own data; all four one-hot patterns are met once per case
    for run_ in range(kr.cdiv(4, nb)):
        cases = [one_hot_case(rng, (run_ * nb + c) % 4, m, n, k) for c in range(nb)]
        res, _ = run(eng, prog, [gemm_inputs(a, b) for a, b in cases])
        for c, ((a, b), out) in enumerate(zip(cases, res)):
            for j, (oa, ob) in enumerate(PAIRS):
                kr.check_gemm_exact(out[j], a, b, f"{name} chain {c} pattern {(run_ * nb + c) % 4} ops {(oa, ob)}")
            check_homogeneity(out, f"{name} chain {c}")
    # accuracy on random floats, then the same chains rotated: each chain's result is bitwise unchanged
    cases = [(rng.normal(size=(m, k)) + 1j * rng.normal(size=(m, k)), rng.normal(size=(k, n)) + 1j * rng.normal(size=(k, n)))
             for _ in range(nb)]
    batch = [gemm_inputs(a, b) for a, b in cases]
    res, _ = run(eng, prog, batch)
    for c, ((a, b), out) in enumerate(zip(cases, res)):
        for j, pair in enumerate(PAIRS):
            if j == 0 or not np.array_equal(out[j], out[0]):
                kr.check_gemm_accuracy(out[j], a, b, f"{name} chain {c} ops {pair}")
        check_homogeneity(out, f"{name} chain {c}")
    if nb > 1:
        rot, _ = run(eng, prog, batch[1:] + batch[:1])
        for c in range(nb):
            for j in range(len(PAIRS)):
                assert np.array_equal(rot[(c - 1) % nb][j], res[c][j]), (name, c, PAIRS[j])


@pytest.mark.parametrize("name", list(kr.GEMM_POISON))
def test_zgemm_poisoned_neighbours(eng, name):
    """every operand between NaN-filled inputs, every C between canaries placed through the free list: the product is
    finite and exact and the canaries are unchanged"""
    m, n, k, nb = kr.GEMM_POISON[name]
    assert (m * k) % 8 == 0 and (k * n) % 8 == 0 and (m * n) % 8 == 0
    r = kr.gemm_route(m, n, k, nb)
    assert (r["tile"], r["fused"]) == kr.GEMM_POISON_EXPECT[name], r
    ins = [("pad0", (PAD,))]
    for o in range(4):
        ins += [(f"A{o}", kr.stored_operand(np.zeros((m, k)), o).shape), (f"padA{o}", (PAD,))]
    for o in range(4):
        ins += [(f"B{o}", kr.stored_operand(np.zeros((k, n)), o).shape), (f"padB{o}", (PAD,))]
    ins += [("canary", (PAD,))]
    holes = []

    def build(p, t):
        canaries = [p.copy(t["canary"])]
        hs = []
        for _ in PAIRS:
            hs.append(p.new((m * n,)))
            canaries.append(p.copy(t["canary"]))
        holes.extend(h.off for h in hs)
        del hs                                     # the products land in these holes: first fit, same size, in order
        cs = [p.matmul(t[f"A{oa}"], t[f"B{ob}"], m, n, k, oa, ob) for oa, ob in PAIRS]
        assert [c.off for c in cs] == holes
        return cs + canaries
    prog = compile_program(ins, build)
    rng = np.random.default_rng(7)
    cases = [(kr.int_complex(rng, (m, k)), kr.int_complex(rng, (k, n))) for _ in range(nb)]
    batch = []
    for a, b in cases:
        d = {nm: np.full(sh, NAN) for nm, sh in ins if nm.startswith("pad")}
        d.update({f"A{o}": kr.stored_operand(a, o) for o in range(4)})
        d.update({f"B{o}": kr.stored_operand(b, o) for o in range(4)})
        d["canary"] = np.full(PAD, CANARY)
        batch.append(d)
    res, _ = run(eng, prog, batch)
    for (a, b), out in zip(cases, res):
        for j, pair in enumerate(PAIRS):
            kr.check_gemm_exact(out[j], a, b, f"poisoned {name} ops {pair}")
        for cn in out[len(PAIRS):]:
            assert np.array_equal(cn, np.full(PAD, CANARY)), f"{name}: a store left its tile"


def test_zgemm_splitk_host_captured_replayed(eng):
    """back-to-back fused split-K products share the tile counters: host-driven, captured and replayed runs of one
    program are bitwise equal and exact"""
    nb = 3
    for m, n, k, oa, ob in kr.SPLITK_CHAIN:
        assert kr.gemm_route(m, n, k, nb)["fused"], (m, n, k)
    ins = []
    for j, (m, n, k, oa, ob) in enumerate(kr.SPLITK_CHAIN):
        ins += [(f"A{j}", kr.stored_operand(np.zeros((m, k)), oa).shape), (f"B{j}", kr.stored_operand(np.zeros((k, n)), ob).shape)]

    def build(p, t):
        return [p.matmul(t[f"A{j}"], t[f"B{j}"], m, n, k, oa, ob) for j, (m, n, k, oa, ob) in enumerate(kr.SPLITK_CHAIN)]
    prog = compile_program(ins, build)
    rng = np.random.default_rng(11)
    data = [[(kr.int_complex(rng, (m, k)), kr.int_complex(rng, (k, n))) for m, n, k, _, _ in kr.SPLITK_CHAIN] for _ in range(nb)]
    batch = [{nm: v for j, (m, n, k, oa, ob) in enumerate(kr.SPLITK_CHAIN)
              for nm, v in ((f"A{j}", kr.stored_operand(d[j][0], oa)), (f"B{j}", kr.stored_operand(d[j][1], ob)))} for d in data]
    host, _ = run(eng, prog, batch)
    g0 = eng.graph_counters()
    eng.graph_policy(0, True)
    try:
        captured, _ = run(eng, prog, batch)
        replayed, _ = run(eng, prog, batch)
    finally:
        eng.graph_policy(1 << 40, False)
    g1 = eng.graph_counters()
    assert g1["graph_captures"] == g0["graph_captures"] + 1 and g1["graph_replays"] == g0["graph_replays"] + 2, (g0, g1)
    for c in range(nb):
        for j in range(len(kr.SPLITK_CHAIN)):
            kr.check_gemm_exact(host[c][j], *data[c][j], f"split-K chain {c} product {j}")
            assert np.array_equal(captured[c][j], host[c][j]) and np.array_equal(replayed[c][j], host[c][j]), (c, j)


# ================================================================================================================ SVD
def svd_program(m, n, keep, nr_bulk):
    """the input between two NaN-filled neighbours (m n is a multiple of 8 in every case here)"""
    ins = [("padL", (PAD,)), ("A", (m, n)), ("padR", (PAD,))]
    return compile_program(ins, lambda p, t: list(p.svd_trunc(t["A"], keep, nr_bulk, 0, 1)))


def counters(eng):
    c = eng.svd_counters()
    return {k: c[k] for k in ("small", "reduced", "subspace", "subspace_fallback", "block_jacobi")}


def run_svd(eng, m, n, keep, mats, nr_bulk=True):
    prog = svd_program(m, n, keep, nr_bulk)
    c0 = counters(eng)
    res, sl = run(eng, prog, [{"padL": np.full(PAD, NAN), "A": a, "padR": np.full(PAD, NAN)} for a in mats])
    c1 = counters(eng)
    return res, sl, {k: c1[k] - c0[k] for k in c0}


def expect_route(delta, route, nb, what):
    assert delta == kr.counter_delta(route, nb), f"{what}: route {route} expected, counters moved {delta}"


def decaying(rng, m, n, d, scale=1.0):
    p = min(m, n)
    s = np.sort(np.exp(-d * np.arange(p)) * (1.0 + 0.2 * rng.random(p)))[::-1]
    return kr.with_spectrum(rng, m, n, s * scale)


@pytest.mark.parametrize("keep", kr.SVD_KEEPS + [kr.SVD_KEEP_EXACT])
def test_svd_subspace_keep_sweep(eng, keep):
    """every block width of the subspace iteration (Cholesky variant, column blocks, the b = 192 cap, keep 100-128 with a
    block narrower than 2 keep, keep = 128 at the edge of the check kernels' row sums) on three chains with different
    spectra; keep 129 takes the exact path"""
    i = (kr.SVD_KEEPS + [kr.SVD_KEEP_EXACT]).index(keep)
    m, n = kr.subspace_shape(keep, ("square", "tall", "wide")[i % 3])
    route = kr.svd_route(m, n, keep)["route"]
    assert route == ("block_jacobi" if keep > 128 else "subspace")
    rng = np.random.default_rng(100 + keep)
    d = kr.subspace_decay(min(keep, 128))
    mats = [decaying(rng, m, n, d * f, sc) for f, sc in ((1.0, 3.7), (0.85, 0.02), (1.2, 55.0))]
    nrb = i % 2 == 0
    res, sl, delta = run_svd(eng, m, n, keep, mats, nrb)
    expect_route(delta, route, 3, f"{m}x{n} keep {keep}")
    for c, (a, (us, vh)) in enumerate(zip(mats, res)):
        kr.check_svd(a, us, vh, sl[c], keep, nrb, what=f"{m}x{n} keep {keep} chain {c}")
    if keep in (49, 100):
        rot, _, _ = run_svd(eng, m, n, keep, mats[1:] + mats[:1], nrb)
        for c in range(3):
            assert all(np.array_equal(x, y) for x, y in zip(rot[(c - 1) % 3], res[c])), f"keep {keep}: chain {c} depends on its place"


@pytest.mark.parametrize("name", list(kr.SVD_SMALL))
def test_svd_small_reduced_variants(eng, name):
    """every one-CTA and cluster variant of the small Jacobi kernel, wide and tall, the reduced path on either side of the
    small kernel's shared-memory limit, and the subspace / exact routes at their neighbouring shapes"""
    m, n, keep = kr.SVD_SMALL[name]
    r = kr.svd_route(m, n, keep)
    assert (r["route"], r.get("kernel")) == kr.SVD_SMALL_EXPECT[name], r
    rng = np.random.default_rng(sum(map(ord, name)))
    if r["route"] == "subspace":
        d = kr.subspace_decay(keep)
        mats = [decaying(rng, m, n, d * f, sc) for f, sc in ((1.0, 1.0), (0.85, 40.0), (1.2, 1e-3))]
    else:
        g = rng.normal(size=(m, n)) + 1j * rng.normal(size=(m, n))
        mats = [g, decaying(rng, m, n, 0.15, 2.5), decaying(rng, m, n, 0.05, 1e-3)]
        mats[2][:, -1] = mats[2][:, 0]               # rank deficient
    res, sl, delta = run_svd(eng, m, n, keep, mats, True)
    expect_route(delta, r["route"], 3, name)
    for c, (a, (us, vh)) in enumerate(zip(mats, res)):
        kr.check_svd(a, us, vh, sl[c], keep, True, what=f"{name} chain {c}")


@pytest.mark.parametrize("kind", kr.SVD_HARD_INPUTS)
@pytest.mark.parametrize("route_name", list(kr.SVD_HARD_ROUTES))
def test_svd_hard_inputs(eng, route_name, kind):
    """repeated singular values across the cut, a flat spectrum, exact rank below keep and between keep and b, the zero
    matrix (finite outputs, slots unchanged), half the rows at 1e-150"""
    m, n, keep = kr.SVD_HARD_ROUTES[route_name]
    route = kr.svd_route(m, n, keep)["route"]
    rng = np.random.default_rng(sum(map(ord, route_name + kind)))
    a = kr.hard_input(rng, kind, m, n, keep) * 1.9
    res, sl, delta = run_svd(eng, m, n, keep, [a], True)
    expect_route(delta, route, 1, f"{route_name} {kind}")
    us, vh = res[0]
    kr.check_svd(a, us, vh, sl[0], keep, True, what=f"{route_name} {kind}")
    if kind == "zero":
        assert not us.any() and np.all(sl[0] == 0)


def homogeneity_inputs(rng, route_name):
    m, n, keep = kr.SVD_HARD_ROUTES[route_name]
    route = kr.svd_route(m, n, keep)["route"]
    if route == "subspace":
        return decaying(rng, m, n, kr.subspace_decay(keep))
    return decaying(rng, m, n, 0.1)


@pytest.mark.parametrize("route_name", list(kr.SVD_HARD_ROUTES))
def test_svd_scale_homogeneity(eng, route_name):
    """svd_trunc(2^+-200 A) = svd_trunc(A) to 1e-13 with the lognorm shifted by +-200 ln 2, on every route"""
    m, n, keep = kr.SVD_HARD_ROUTES[route_name]
    route = kr.svd_route(m, n, keep)["route"]
    rng = np.random.default_rng(sum(map(ord, route_name)))
    a = homogeneity_inputs(rng, route_name)
    mats = [a, a * 2.0 ** 200, a * 2.0 ** -200]
    res, sl, delta = run_svd(eng, m, n, keep, mats, True)
    expect_route(delta, route, 3, route_name)
    kr.check_svd(a, *res[0], sl[0], keep, True, what=route_name)
    p0 = res[0][0] @ res[0][1]
    for c, e in ((1, 200), (2, -200)):
        us, vh = res[c]
        assert np.all(np.isfinite(us)) and np.all(np.isfinite(vh)), (route_name, e)
        assert np.linalg.norm(us @ vh - p0) <= 1e-13 * np.linalg.norm(p0), (route_name, e, np.linalg.norm(us @ vh - p0) / np.linalg.norm(p0))
        assert abs(sl[c, 0] - sl[0, 0] - e * np.log(2.0)) <= 1e-12 * abs(e * np.log(2.0)), (route_name, e, sl[c, 0], sl[0, 0])
        assert abs(sl[c, 1] - sl[0, 1]) <= 1e-12 and sl[c, -1] == 0, (route_name, e, sl[c])


@pytest.mark.parametrize("route_name", list(kr.SVD_HARD_ROUTES))
def test_svd_extreme_scales(eng, route_name, record_property):
    """2^300, 2^-300 and 1e-150 times an O(1) matrix, once per route.  No route holds there (DESIGN.md, scale range of the
    truncated SVD: the Jacobi rotations and the subspace Gram matrix form fourth powers of the scale), and real programs stay
    far inside 2^+-150 (test_kernel_routes_cpu.py).  What each route gives is recorded, not asserted."""
    m, n, keep = kr.SVD_HARD_ROUTES[route_name]
    rng = np.random.default_rng(sum(map(ord, route_name)) + 1)
    a = homogeneity_inputs(rng, route_name)
    scales = [1.0, 2.0 ** 300, 2.0 ** -300, 1e-150]
    res, sl, _ = run_svd(eng, m, n, keep, [a * s for s in scales], True)
    p0 = res[0][0] @ res[0][1]
    rec = {}
    for c, s in enumerate(scales[1:], 1):
        us, vh = res[c]
        finite = bool(np.all(np.isfinite(us)) and np.all(np.isfinite(vh)))
        err = float(np.linalg.norm(np.nan_to_num(us @ vh) - p0) / np.linalg.norm(p0))
        rec[f"{s:.3g}"] = {"finite": finite, "rel_err": err, "lognorm_err": float(sl[c, 0] - sl[0, 0] - np.log(s)),
                           "trunc": float(sl[c, 1]), "status": float(sl[c, -1])}
    print(f"extreme scales {route_name}: {rec}")
    record_property("extreme_scales", rec)


# ================================================================================================================ QR
@pytest.mark.parametrize("m,n", list(kr.QR_CASES))
def test_qr_routes_poisoned(eng, m, n):
    """Cholesky-QR2, blocked Gram-Schmidt and Householder at their edges, input between NaN-filled neighbours"""
    ins = [("padL", (PAD,)), ("A", (m, n)), ("padR", (PAD,))]
    prog = compile_program(ins, lambda p, t: list(p.qr(t["A"])))
    rng = np.random.default_rng(m * 1000 + n)
    mats = [rng.normal(size=(m, n)) + 1j * rng.normal(size=(m, n)) for _ in range(2)]
    mats[1][:, -1] = mats[1][:, 0]
    res, _ = run(eng, prog, [{"padL": np.full(PAD, NAN), "A": a, "padR": np.full(PAD, NAN)} for a in mats])
    k = min(m, n)
    for a, (q, r) in zip(mats, res):
        assert np.all(np.isfinite(q)) and np.all(np.isfinite(r)), (m, n)
        assert np.linalg.norm(q @ r - a) <= 1e-13 * np.linalg.norm(a), (m, n)
        assert np.linalg.norm(q.conj().T @ q - np.eye(k)) <= 1e-13 * k, (m, n)
        assert np.allclose(np.tril(r, -1), 0), (m, n)
