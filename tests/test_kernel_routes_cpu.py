"""CPU tier of the kernel-route tests: the dispatch mirror reaches every reachable kernel instantiation with the cases the
GPU tier runs, the reference checkers reject near-miss results, and the SVD inputs of real programs stay inside the
scale range the SVD routes hold (DESIGN.md, scale range of the truncated SVD)."""
import numpy as np
import pytest

import kernel_routes as kr


# ------------------------------------------------------------------------------------------------ route table
def test_route_table_is_complete():
    reached = kr.reached_instantiations()
    assert reached == kr.INSTANTIATIONS, (sorted(kr.INSTANTIATIONS - reached), sorted(reached - kr.INSTANTIATIONS))
    assert not (kr.INSTANTIATIONS & kr.UNREACHABLE)


def test_mirror_puts_every_case_where_the_table_says():
    for name, (m, n, k, nb) in kr.GEMM_CASES.items():
        r = kr.gemm_route(m, n, k, nb)
        assert (r["tile"], r["fused"], r["rows_on_x"]) == kr.GEMM_EXPECT[name], (name, r)
        assert m % r["tile"] and n % r["tile"] and k % 16, name
    assert {kr.GEMM_EXPECT[nm][2] for nm in kr.GEMM_CASES if kr.GEMM_EXPECT[nm][0] in (32, 64)} == {True, False}
    assert {kr.GEMM_CASES[nm][3] for nm in kr.GEMM_CASES} >= {1, 3, 37}
    assert any(k < 16 for _, _, k, _ in kr.GEMM_CASES.values())
    for name, (m, n, k, nb) in kr.GEMM_POISON.items():
        r = kr.gemm_route(m, n, k, nb)
        assert (r["tile"], r["fused"]) == kr.GEMM_POISON_EXPECT[name], (name, r)
    for m, n, k, _, _ in kr.SPLITK_CHAIN:
        assert kr.gemm_route(m, n, k, 3)["fused"]
    for name, (m, n, keep) in kr.SVD_SMALL.items():
        r = kr.svd_route(m, n, keep)
        assert (r["route"], r.get("kernel")) == kr.SVD_SMALL_EXPECT[name], (name, r)
    blocks = set()
    for keep in kr.SVD_KEEPS:
        for kind in ("square", "tall", "wide"):
            m, n = kr.subspace_shape(keep, kind)
            r = kr.svd_route(m, n, keep)
            assert r["route"] == "subspace" and min(m, n) >= 1.25 * r["b"], (keep, kind, r)
            blocks.add(r["b"])
    assert {b for b in blocks if b <= 32} and {104, 112} <= blocks and 192 in blocks
    assert kr.svd_route(*kr.subspace_shape(128, "square"), kr.SVD_KEEP_EXACT)["route"] == "block_jacobi"
    assert kr.svd_route(*kr.subspace_shape(100, "square"), 100)["it_max"] == 72        # block narrower than 2 keep
    for (m, n), route in kr.QR_CASES.items():
        assert kr.qr_route(m, n) == route, (m, n)
    assert {r["route"] for r in (kr.svd_route(*v) for v in kr.SVD_HARD_ROUTES.values())} == {"small", "reduced", "subspace", "block_jacobi"}


def test_unreachable_instantiations_stay_unreachable():
    """no shape the small-SVD dispatch accepts, and no Rayleigh-Ritz block, lands on an instantiation listed as unreachable"""
    seen = set()
    for p in range(1, 129):
        for q in range(p, 1400):
            for m, n in ((p, q), (q, p)):
                if kr.svd_small_fits(m, n):
                    seen.add(kr.small_kernel(m, n))
    for b in range(8, 193, 8):
        seen.add(kr.small_kernel(b, b))
    assert not (seen & kr.UNREACHABLE), seen & kr.UNREACHABLE
    assert {x for x in kr.INSTANTIATIONS if x[0] in ("svd_small", "svd_cluster")} <= seen


# ------------------------------------------------------------------------------------------------ checkers reject near misses
def _ops_case(rng, m, n, k):
    a, b = kr.int_complex(rng, (m, k)), kr.int_complex(rng, (k, n))
    return a, b


def test_gemm_checkers_reject_a_dropped_k_slab_and_a_flipped_conjugation():
    rng = np.random.default_rng(3)
    for m, n, k in ((20, 12, 37), (5, 7, 33), (16, 16, 17)):
        a, b = _ops_case(rng, m, n, k)
        good = kr.exact_product(a, b)
        kr.check_gemm_exact(good, a, b)
        kr.check_gemm_accuracy(good, a, b)
        k0 = (k - 1) // 16 * 16                          # start of the last k-slab
        dropped = kr.exact_product(a[:, :k0], b[:k0])
        flipped = kr.exact_product(np.conj(a), b)
        for bad in (dropped, flipped):
            with pytest.raises(AssertionError):
                kr.check_gemm_exact(bad, a, b)
            with pytest.raises(AssertionError):
                kr.check_gemm_accuracy(bad, a, b)
        af, bf = a + 0.3 * rng.normal(size=a.shape), b + 0.2j * rng.normal(size=b.shape)
        ref = (af.astype(np.clongdouble) @ bf.astype(np.clongdouble)).astype(np.complex128)
        kr.check_gemm_accuracy(ref, af, bf)
        for bad in (af[:, :k0] @ bf[:k0], np.conj(af) @ bf):
            with pytest.raises(AssertionError):
                kr.check_gemm_accuracy(bad, af, bf)


def _lapack_trunc(a, keep, nr_bulk):
    u, s, vh = np.linalg.svd(a, full_matrices=False)
    fro = np.linalg.norm(s)
    f = fro if (nr_bulk and fro > 0) else 1.0
    sl = np.zeros(8)
    if fro > 0:
        sl[1] = np.sqrt(np.sum(s[keep:] ** 2) / np.sum(s ** 2))
        sl[0] = np.log(fro) if nr_bulk else 0.0
    return u[:, :keep] * s[:keep] / f, vh[:keep].copy(), sl, u, s, vh


@pytest.mark.parametrize("nr_bulk", [True, False])
def test_svd_checker_accepts_lapack_and_rejects_near_misses(nr_bulk):
    rng = np.random.default_rng(5)
    m, n, keep = 60, 40, 10
    s = np.exp(-0.2 * np.arange(40))
    s[7:10] = s[7]                                       # degenerate cluster inside the kept part, at 7, 8, 9
    s[10:13] = s[10]
    a = kr.with_spectrum(rng, m, n, s) * 3.0
    us, vh, sl, u, sv, vv = _lapack_trunc(a, keep, nr_bulk)
    f = np.linalg.norm(sv) if nr_bulk else 1.0
    kr.check_svd(a, us, vh, sl, keep, nr_bulk)
    for kind in ("zero", "rank_below_keep", "repeated_at_cut", "flat", "tiny_rows"):
        h = kr.hard_input(rng, kind, m, n, keep)
        kr.check_svd(h, *_lapack_trunc(h, keep, nr_bulk)[:3], keep, nr_bulk)
    # one US column replaced by the other member's direction of the degenerate cluster (same norm)
    bad = us.copy()
    bad[:, 8] = u[:, 9] * sv[8] / f
    with pytest.raises(kr.SvdCheckError, match="Eckart-Young"):
        kr.check_svd(a, bad, vh, sl, keep, nr_bulk)
    # a wrong singular value
    bad = us.copy()
    bad[:, 3] *= 1 + 1e-8
    with pytest.raises(kr.SvdCheckError, match="column norms|Eckart-Young"):
        kr.check_svd(a, bad, vh, sl, keep, nr_bulk)
    # Vh rows not orthonormal, product and column norms unchanged: Vh' = M Vh, US' = US M^-1
    eps = 1e-6
    vb, ub = vh.copy(), us.copy()
    vb[0] += eps * vh[1]
    ub[:, 1] -= eps * us[:, 0]
    with pytest.raises(kr.SvdCheckError, match="Vh orthonormal"):
        kr.check_svd(a, ub, vb, sl, keep, nr_bulk)
    # slots
    for j, delta in ((1, 1e-9), (0, 1e-9), (-1, 1.0)):
        if j == 0 and not nr_bulk:
            continue
        s2 = sl.copy()
        s2[j] += delta
        with pytest.raises(kr.SvdCheckError, match="slot"):
            kr.check_svd(a, us, vh, s2, keep, nr_bulk)
    bad = us.copy()
    bad[0, 0] = np.nan
    with pytest.raises(kr.SvdCheckError, match="non-finite"):
        kr.check_svd(a, bad, vh, sl, keep, nr_bulk)


# ------------------------------------------------------------------------------------------------ SVD input norm survey
SURVEY_LIMIT = 2.0 ** 150


@pytest.fixture
def svd_norms():
    from np_vm import NumpyEngine
    NumpyEngine.svd_input_norms = []
    yield NumpyEngine.svd_input_norms
    NumpyEngine.svd_input_norms = None


def _check_norms(norms, what):
    x = np.array([v for v in norms if v > 0])
    assert len(x), what
    lo, hi = x.min(), x.max()
    print(f"SVD input survey {what}: {len(norms)} truncations, |A|_F in [{lo:.3e}, {hi:.3e}] (2^{np.log2(lo):.1f} .. 2^{np.log2(hi):.1f})")
    assert 1.0 / SURVEY_LIMIT <= lo and hi <= SURVEY_LIMIT, (what, lo, hi)


@pytest.mark.parametrize("D", [2, 3, 4])
def test_svd_input_norms_of_bp(vm_engines, svd_norms, D):
    """the block-BP programs of the golden runs (D = 2, 3, 4, N = 2) on the op-stream interpreter"""
    import os
    from conftest import GOLDEN
    from kagomeperiodicbp_b200 import belief_propagation as bp
    from kagomeperiodicbp_b200.containers import BPConfig, UnitCell
    g = np.load(os.path.join(GOLDEN, f"bp_D{D}_N2_damp.npz"))
    cell = UnitCell(g["A"], g["B"], g["C"])
    tn = bp.KagomeTNRepeatedUnitCell(cell, 2)
    tn.connect_uniform_messages()
    cfg = BPConfig(trunc_dim=2 * D * D, msg_diff_terminate=1e-6, damping=0.1, init_msg="UQ", max_iterations=3)
    bp.belief_propagation(tn, tn.messages, cfg)
    _check_norms(svd_norms, f"BP D={D}")


def test_svd_input_norms_of_chain_and_ite(vm_engines, svd_norms, monkeypatch):
    """one boundary-MPS chain contraction and one whole ITE step (ToCore chains, edge environment, gate + ALS)"""
    from np_vm import NumpyEngine
    import kagomeperiodicbp_b200.linalg as linalg
    from kagomeperiodicbp_b200 import ite_flow
    import test_cpu_tier
    test_cpu_tier.test_bubblecon_api_via_interpreter(vm_engines)
    _check_norms(svd_norms, "chain D=2")
    engines = {}
    monkeypatch.setattr(linalg, "get_engine", lambda key="default", device=0: engines.setdefault(key, NumpyEngine()))
    monkeypatch.setattr(ite_flow, "_backend", linalg.ResidentBackend("vm-ite", arena_elems=1 << 23))
    import test_ite_flow_gpu
    del svd_norms[:]
    test_ite_flow_gpu.test_full_ite_step_matches_oracle()
    _check_norms(svd_norms, "ITE step D=2")
