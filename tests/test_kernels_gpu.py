"""GPU tier: every device op of the C ABI against numpy on seeded inputs (complex128, tolerance stated per test)."""
import numpy as np
import pytest

from kagomeperiodicbp_b200.program import Program
from kagomeperiodicbp_b200.runtime import Compiled

pytestmark = pytest.mark.gpu

rng = np.random.default_rng(1234)


def rnd(*s):
    return rng.normal(size=s) + 1j * rng.normal(size=s)


@pytest.fixture(scope="module")
def eng():
    from kagomeperiodicbp_b200.engine import Engine
    e = Engine(0)
    yield e
    e.close()


def run(eng, build, batch_inputs, n_slots=8):
    p = Program(n_slots)
    first = batch_inputs[0]
    dts = [(f"i{k}", p.input(f"i{k}", a.shape)) for k, a in enumerate(first)]
    outs = build(p, [t for _, t in dts])
    comp = Compiled(p, dts, [(f"o{k}", t) for k, t in enumerate(outs)])
    o, sl, rc = comp.run(eng, [{f"i{k}": a for k, a in enumerate(ins)} for ins in batch_inputs])
    return [[oc[f"o{k}"] for k in range(len(outs))] for oc in o], sl


@pytest.mark.parametrize("shape,perm", [((2, 3, 4), (2, 0, 1)), ((4, 4, 4, 4), (3, 1, 0, 2)), ((2, 1, 3, 5), (3, 2, 1, 0)),
                                        ((32, 4, 4, 4, 4, 32), (0, 2, 4, 5, 1, 3)), ((7,), (0,))])
def test_permute(eng, shape, perm):
    xs = [[rnd(*shape)] for _ in range(3)]
    for cj in (False, True):
        res, _ = run(eng, lambda p, t: [p.transpose(t[0], perm, conj=cj) if (cj or list(perm) != list(range(len(perm)))) else p.copy(t[0])], xs)
        for (x,), (r,) in zip(xs, res):
            e = x.transpose(perm)
            e = np.conj(e) if cj else e
            assert np.array_equal(r, e)   # pure data movement: bit exact


@pytest.mark.parametrize("m,n,k", [(1, 1, 1), (3, 5, 7), (64, 64, 16), (65, 63, 17), (162, 81, 9), (128, 32, 512), (1, 1, 300), (200, 130, 70)])
def test_gemm_all_ops(eng, m, n, k):
    for oa in range(4):
        for ob in range(4):
            sa = (m, k) if oa in (0, 3) else (k, m)
            sb = (k, n) if ob in (0, 3) else (n, k)
            batch = [[rnd(*sa), rnd(*sb)] for _ in range(2)]
            res, _ = run(eng, lambda p, t: [p.matmul(t[0], t[1], m, n, k, oa, ob)], batch)
            for (a, b), (r,) in zip(batch, res):
                A = a if oa in (0, 3) else a.T
                A = np.conj(A) if oa in (2, 3) else A
                B = b if ob in (0, 3) else b.T
                B = np.conj(B) if ob in (2, 3) else B
                e = A @ B
                assert np.linalg.norm(r - e) <= 1e-13 * max(1.0, np.linalg.norm(e)), (m, n, k, oa, ob)


def test_tensordot_conj(eng):
    a, b = rnd(6, 2, 2, 5), rnd(2, 2, 3, 2)
    res, _ = run(eng, lambda p, t: [p.tensordot(t[0], t[1], ([1, 2], [3, 0]), conj_b=True)], [[a, b]])
    e = np.tensordot(a, np.conj(b), axes=([1, 2], [3, 0]))
    assert np.allclose(res[0][0], e, atol=1e-13)


@pytest.mark.parametrize("m,n", [(5, 3), (3, 5), (16, 16), (162, 18), (18, 162), (512, 32), (64, 64), (1, 4), (4, 1), (256, 32), (768, 48),
                                 (243, 27), (256, 16), (130, 7), (1024, 40), (1100, 16), (96, 200),
                                 (1024, 64), (2592, 72), (2000, 40), (1300, 130),        # TSQR over row blocks / one-CTA kernel
                                 (672, 672), (392, 392), (816, 264),                      # large, not skinny: block Gram-Schmidt over tall-skinny blocks
                                 (300, 200), (700, 129), (384, 384),                      # too little workspace for the blocked path: Householder
                                 (208, 32), (207, 32), (592, 96), (584, 96), (300, 8), (300, 7)])   # Cholesky-QR2 at its workspace and width edges
def test_qr(eng, m, n):
    batch = [[rnd(m, n)] for _ in range(3)]
    # make one of them rank deficient
    batch[1][0][:, -1] = batch[1][0][:, 0]
    batch[2][0][:] = 0
    batch[2][0][0, 0] = 1.0
    res, _ = run(eng, lambda p, t: list(p.qr(t[0])), batch)
    k = min(m, n)
    for (a,), (q, r) in zip(batch, res):
        assert q.shape == (m, k) and r.shape == (k, n)
        assert np.linalg.norm(q @ r - a) <= 1e-13 * max(1.0, np.linalg.norm(a))
        assert np.linalg.norm(q.conj().T @ q - np.eye(k)) <= 1e-13 * k
        assert np.allclose(np.tril(r, -1), 0)


def test_qr_tiny_scale(eng):
    """columns at 1e-150 (rows the truncation emptied) must not underflow in the norms (bmpslib keeps such tensors alive)"""
    for m, n in [(512, 32), (64, 16)]:
        a = rnd(m, n)
        a[:, n // 2:] *= 1e-150
        res, _ = run(eng, lambda p, t: list(p.qr(t[0])), [[a]])
        q, r = res[0]
        assert np.linalg.norm(q.conj().T @ q - np.eye(n)) <= 1e-13 * n
        d = q @ r - a
        assert np.linalg.norm(d[:, :n // 2]) <= 1e-13 * np.linalg.norm(a)
        assert np.linalg.norm(d[:, n // 2:]) <= 1e-13 * np.linalg.norm(a[:, n // 2:])


def test_lq(eng):
    a = rnd(18, 162)
    res, _ = run(eng, lambda p, t: list(p.lq(t[0])), [[a]])
    l, q = res[0]
    assert l.shape == (18, 18) and q.shape == (18, 162)
    assert np.linalg.norm(l @ q - a) <= 1e-13 * np.linalg.norm(a)
    assert np.linalg.norm(q @ q.conj().T - np.eye(18)) <= 1e-12


@pytest.mark.parametrize("m,n,keep", [(32, 32, 8), (8, 32, 8), (32, 8, 4), (162, 162, 18), (81, 162, 18), (162, 81, 18),
                                      (100, 37, 37), (512, 512, 32), (256, 512, 32), (5, 3, 2), (1, 7, 1)])
def test_svd_truncate(eng, m, n, keep):
    batch = []
    for c in range(3):
        a = rnd(m, n)
        if c == 1:   # decaying spectrum like a boundary MPS
            u, s, vh = np.linalg.svd(a, full_matrices=False)
            a = (u * (2.0 ** -np.arange(len(s)))) @ vh
        if c == 2 and min(m, n) > 2:   # rank deficient
            a[:, -1] = a[:, 0]
            a[-1, :] = a[0, :]
        batch.append([a])
    for nrb in (0, 1):
        res, sl = run(eng, lambda p, t: list(p.svd_trunc(t[0], keep, bool(nrb), 0, 1)), batch)
        for c, ((a,), (us, vh)) in enumerate(zip(batch, res)):
            u, s, v = np.linalg.svd(a, full_matrices=False)
            fro = np.linalg.norm(s)
            ref = (u[:, :keep] * s[:keep]) @ v[:keep]
            scale = fro if nrb else 1.0
            got = (us @ vh) * scale
            gap_ok = keep == len(s) or s[keep - 1] - s[keep] > 1e-6 * s[0]
            if gap_ok:
                assert np.linalg.norm(got - ref) <= 1e-11 * fro, (m, n, keep, c, nrb)
            # V^H rows orthonormal where the singular value is not negligible
            big = s[:keep] > 1e-10 * s[0]
            gram = (vh @ vh.conj().T)[np.ix_(big, big)]
            assert np.linalg.norm(gram - np.eye(big.sum())) <= 1e-10, (m, n, keep, c)
            terr = np.sqrt(np.sum(s[keep:] ** 2) / np.sum(s ** 2))
            assert abs(sl[c, 1] - terr) <= 1e-10
            if nrb:
                assert abs(sl[c, 0] - np.log(fro)) <= 1e-12 * max(1, abs(np.log(fro)))
            sv = np.sort(np.linalg.norm(us, axis=0))[::-1] * scale
            assert np.allclose(sv, s[:keep], rtol=1e-10, atol=1e-12 * s[0])


@pytest.mark.parametrize("m,n,keep,decay", [(512, 512, 32, 0.08), (256, 512, 32, 0.1), (512, 256, 32, 0.1), (256, 256, 32, 0.12),
                                            (162, 162, 18, 0.15), (300, 200, 20, 0.2), (512, 512, 32, 0.03)])
def test_svd_subspace_path(eng, m, n, keep, decay):
    """boundary-MPS-like spectra (s_j ~ exp(-decay j), near-degenerate cut): the subspace-iteration path must take
    them (no fallback) and reproduce the exact rank-`keep` truncation."""
    batch = []
    for c in range(2):
        a = rnd(m, n)
        u, s, vh = np.linalg.svd(a, full_matrices=False)
        s = np.exp(-decay * np.arange(len(s))) * (1.0 + 0.3 * rng.random(len(s)))
        s = np.sort(s)[::-1]
        if c == 1:
            s[keep] = s[keep - 1] * 0.99       # 1 % gap at the cut
        batch.append([(u * s) @ vh * 3.7])
    before = eng.svd_counters()
    res, sl = run(eng, lambda p, t: list(p.svd_trunc(t[0], keep, True, 0, 1)), batch)
    after = eng.svd_counters()
    if decay >= 0.05:
        # counted per chain by the device-side decision kernel
        assert after["subspace"] == before["subspace"] + len(batch) and after["subspace_fallback"] == before["subspace_fallback"], (before, after)
    for c, ((a,), (us, vh)) in enumerate(zip(batch, res)):
        u, s, v = np.linalg.svd(a, full_matrices=False)
        fro = np.linalg.norm(s)
        ref = (u[:, :keep] * s[:keep]) @ v[:keep]
        got = (us @ vh) * fro
        gap = (s[keep - 1] - s[keep]) / s[0]
        assert np.linalg.norm(got - ref) <= 2e-13 * fro / gap, (m, n, keep, c, np.linalg.norm(got - ref) / fro, gap)
        assert np.linalg.norm(vh @ vh.conj().T - np.eye(keep)) <= 1e-12
        terr = np.sqrt(np.sum(s[keep:] ** 2) / np.sum(s ** 2))
        assert abs(sl[c, 1] - terr) <= 1e-10
        assert abs(sl[c, 0] - np.log(fro)) <= 1e-12 * max(1, abs(np.log(fro)))
        assert sl[c, -1] == 0


def test_normalize_embed_eye(eng):
    a, b = rnd(3, 4, 5), rnd(2, 4, 6)

    def build(p, t):
        x = p.copy(t[0])
        p.normalize_(x, 2)
        s = p.zeros((5, 4, 11))
        p.embed(s, (0, 0, 0), t[0], 0.9)
        p.embed(s, (3, 0, 5), t[1], -0.1 + 0.2j)
        return [x, s, p.eye(6, 6)]
    res, sl = run(eng, build, [[a, b]])
    x, s, e = res[0]
    assert np.allclose(x, a / np.linalg.norm(a), atol=1e-15)
    assert abs(sl[0, 2] - np.log(np.linalg.norm(a))) < 1e-13
    ref = np.zeros((5, 4, 11), complex)
    ref[:3, :, :5] = 0.9 * a
    ref[3:, :, 5:] = (-0.1 + 0.2j) * b
    assert np.allclose(s, ref, atol=1e-15)
    assert np.array_equal(e, np.eye(6))


@pytest.mark.parametrize("m,n,keep", [(800, 800, 72), (1296, 648, 82)])
def test_svd_subspace_wide_block_two_column_blocks(eng, m, n, keep):
    """keep = 72 / 82 (chi_bp and chi at D = 6): block of 144 / 168 columns, wider than one CTA's Cholesky takes -- the panel is
    orthogonalised as two column blocks (block Gram-Schmidt + Cholesky-QR per block)."""
    a = rnd(m, n)
    u, s, vh = np.linalg.svd(a, full_matrices=False)
    s = np.exp(-0.04 * np.arange(len(s)))
    a = (u * s) @ vh
    before = eng.svd_counters()
    res, sl = run(eng, lambda p, t: list(p.svd_trunc(t[0], keep, True, 0, 1)), [[a]])
    after = eng.svd_counters()
    assert after["subspace"] == before["subspace"] + 1 and after["subspace_fallback"] == before["subspace_fallback"], (before, after)
    us, v = res[0]
    ref = (u[:, :keep] * s[:keep]) @ vh[:keep]
    gap = (s[keep - 1] - s[keep]) / s[0]
    assert np.linalg.norm(us @ v * np.linalg.norm(s) - ref) <= 2e-13 * np.linalg.norm(s) / gap
    assert np.linalg.norm(v @ v.conj().T - np.eye(keep)) <= 1e-12
    assert abs(sl[0, 1] - np.sqrt(np.sum(s[keep:] ** 2) / np.sum(s ** 2))) <= 1e-10 and sl[0, -1] == 0


def test_svd_subspace_widest_block(eng):
    """keep = 42 (chi = 2 D^2 + 10 at D = 4: the ToCore / ToEdge chains) runs the subspace path with a block of 88 columns
    (the register Cholesky of up to 96 columns).  The widest one-block panel (112, chol_blocked_kernel) is reached by keep 49-56
    in test_kernel_routes_gpu.py."""
    m, n, keep = 672, 672, 42
    a = rnd(m, n)
    u, s, vh = np.linalg.svd(a, full_matrices=False)
    s = np.exp(-0.07 * np.arange(len(s)))
    a = (u * s) @ vh
    before = eng.svd_counters()
    res, sl = run(eng, lambda p, t: list(p.svd_trunc(t[0], keep, True, 0, 1)), [[a]])
    after = eng.svd_counters()
    assert after["subspace"] == before["subspace"] + 1
    us, v = res[0]
    ref = (u[:, :keep] * s[:keep]) @ vh[:keep]
    assert np.linalg.norm(us @ v * np.linalg.norm(s) - ref) <= 1e-11 * np.linalg.norm(s)
