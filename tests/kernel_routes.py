"""Pure-Python mirror of the host dispatch that picks a kernel instantiation by shape, the reference checkers of the
kernel-route tests, and their case tables.  Nothing here touches a device: the CPU tier checks the mirror and the
checkers, the GPU tier (test_kernel_routes_gpu.py) runs the cases.

Every rule below is a copy of a host function in kagomeperiodicbp_b200/csrc and names it.  If the C++ dispatch changes,
the mirror must change with it; test_kernel_routes_cpu.py then shows which case no longer reaches its kernel.

Reachable instantiations and the case that reaches each (``INSTANTIATIONS`` is the table the CPU tier checks):

    zgemm_dmma_kernel<16,16,3,2,A_KC,B_KC>   (4 layouts)  GEMM_CASES "16", "16f" (fused split-K), ZGEMM_POISON, SPLITK_CHAIN
    zgemm_dmma_kernel<32,32,4,8,A_KC,B_KC>   (4 layouts)  GEMM_CASES "32", "32x"
    zgemm_dmma_kernel<64,64,3,8,A_KC,B_KC>   (4 layouts)  GEMM_CASES "64", "64x"
    svd_small_kernel<true,32>                SVD_SMALL "40x100"
    svd_small_kernel<false,32>               SVD_SMALL "20x600", "600x20"
    svd_small_kernel<false,16>               SVD_SMALL "65x200", "130x65"
    svd_cluster_kernel<2..6,8>  wide         SVD_SMALL "48x60", "50x90", "60x120", "64x150", "81x162"
    svd_cluster_kernel<4..6,8>  tall         SVD_SMALL "60x48", "100x50", "130x60"
    reduced (Householder QR + small kernel)  SVD_SMALL "32x449", "417x32"
    chol_reg_kernel<1>                       SVD_KEEPS keep 8, 16 (b <= 32); keep 57-64 as second column block
    chol_reg_kernel<2>                       SVD_KEEPS keep 17, 32 (b <= 64)
    chol_reg_kernel<3>                       SVD_KEEPS keep 33, 48 (b <= 96), first block of every wide panel
    chol_blocked_kernel                      SVD_KEEPS keep 49, 56 (b = 104, 112)
    two column blocks 96 + b2                SVD_KEEPS keep 57 .. 128, the b = 192 cap from keep 92 on
    block-Jacobi exact path                  SVD_KEEPS keep 129; SVD_SMALL "200x160"
    qr: cholqr2 / blocked / Householder      QR_CASES

Unreachable (compiled, and given shared-memory attributes, but no shape reaches them through the dispatch):

    svd_small_kernel<*,8>       a group of 8 lanes means more than 64 row pairs, i.e. p > 128, which svd_small_fits refuses;
                                the Rayleigh-Ritz call (p = b <= 192) takes the cluster kernel.  Only a refused cluster
                                launch falls back to it.
    svd_small_kernel<true,16>   16 lanes need p > 64 (or a failed cluster test, q > 192), cached needs q <= 96 >= p.
    svd_cluster_kernel<1,8>     one column per lane means q <= 32 < 48 <= p.
"""
from __future__ import annotations

import numpy as np


def cdiv(a, b):
    return -(-int(a) // int(b))


def rup8(x):
    return cdiv(x, 8) * 8


# ---------------------------------------------------------------------------------------------------------------- ZGEMM
GEMM_BK = 16                 # k_gemm.cu: BK
GEMM_MAX_TILES = 4096        # k_gemm.cu: GEMM_MAX_TILES
GEMM_WARPS_TARGET = 900      # k_gemm.cu: GEMM_WARPS_TARGET
GEMM_SCRATCH = 1 << 20       # kbp_capi.cu: KBP_GEMM_SCRATCH (split-K partials per chain)
OP_N, OP_T, OP_C, OP_J = 0, 1, 2, 3


def gemm_route(m, n, k, nb, ksplit=0):
    """k_gemm.cu: gemm_splitk (automatic split-K, tile choice) and launch_gemm_l (grid orientation).  ``ksplit`` = 0 is
    the automatic choice every OP_GEMM takes."""
    ks, fused = max(ksplit, 1), False
    if ksplit == 0:
        tiles16 = cdiv(n, 16) * cdiv(m, 16)
        warps = 2 * tiles16 * nb
        slabs = cdiv(k, GEMM_BK)
        ks = 1
        if warps < 600 and slabs >= 8 and tiles16 <= GEMM_MAX_TILES:
            ks = cdiv(GEMM_WARPS_TARGET, warps)
            ks = min(ks, slabs // 4, 16)
            while ks > 1 and ks * m * n > GEMM_SCRATCH:
                ks -= 1
        ks = max(ks, 1)
        fused = ks > 1
    ctas64 = cdiv(n, 64) * cdiv(m, 64) * nb * ks
    ctas32 = cdiv(n, 32) * cdiv(m, 32) * nb * ks
    tile = 16 if (fused or ctas32 < 96) else (64 if ctas64 >= 96 else 32)
    return {"tile": tile, "ksplit": ks, "fused": fused, "rows_on_x": cdiv(m, tile) > cdiv(n, tile)}


def gemm_layout(opA, opB):
    """k_gemm.cu: launch_gemm -- (A k-contiguous, B k-contiguous) template arguments."""
    return (opA in (OP_N, OP_J), opB in (OP_T, OP_C))


def gemm_kernel(m, n, k, nb, opA, opB):
    r = gemm_route(m, n, k, nb)
    return ("zgemm", r["tile"]) + gemm_layout(opA, opB)


# GEMM route cases: name -> (m, n, k, nb).  m, n are not multiples of the tile, k % 16 != 0, both grid orientations.
GEMM_CASES = {
    "16": (65, 63, 17, 1),           # plain 16 x 16, rows on x
    "16y": (13, 40, 7, 3),           # plain 16 x 16, columns on x, k < 16
    "16f": (40, 40, 1000, 1),        # fused split-K, ks = 15
    "16fy": (24, 56, 777, 3),        # fused split-K on 3 chains, columns on x
    "32": (520, 130, 45, 2),         # 32 x 32, rows on x
    "32x": (300, 200, 37, 2),        # 32 x 32, rows on x, k = 37
    "32y": (100, 330, 31, 3),        # 32 x 32, columns on x
    "64": (300, 20, 9, 37),          # 64 x 64 on 37 chains, rows on x
    "64x": (250, 600, 33, 3),        # 64 x 64, columns on x
    "64n": (600, 650, 20, 1),        # 64 x 64 on one chain, columns on x
}
GEMM_EXPECT = {"16": (16, False, True), "16y": (16, False, False), "16f": (16, True, False), "16fy": (16, True, False),
               "32": (32, False, True), "32x": (32, False, True), "32y": (32, False, False),
               "64": (64, False, True), "64x": (64, False, False), "64n": (64, False, False)}       # (tile, fused, rows_on_x)

# operands surrounded by NaN-filled inputs: m k, k n and m n are multiples of 8, so no zero gap sits between them
GEMM_POISON = {"16": (20, 12, 10, 1), "16f": (20, 12, 250, 1), "32": (200, 120, 9, 4), "64": (200, 120, 9, 12)}
GEMM_POISON_EXPECT = {"16": (16, False), "16f": (16, True), "32": (32, False), "64": (64, False)}

# back-to-back fused split-K products of one program: (m, n, k, opA, opB)
SPLITK_CHAIN = [(40, 40, 1000, OP_N, OP_N), (40, 40, 1000, OP_C, OP_N), (24, 56, 777, OP_N, OP_T), (40, 40, 1000, OP_J, OP_C)]


def stored_operand(x, op):
    """what to store so that op(stored) == x (k_gemm.cu op codes: N, T, C = conjugate transpose, J = conjugate)."""
    if op == OP_N:
        return x
    if op == OP_T:
        return np.ascontiguousarray(x.T)
    if op == OP_C:
        return np.ascontiguousarray(np.conj(x).T)
    return np.conj(x)


def int_complex(rng, shape, lo=-8, hi=8):
    return rng.integers(lo, hi + 1, size=shape).astype(np.float64) + 1j * rng.integers(lo, hi + 1, size=shape)


def exact_product(a, b):
    """integer-valued complex operands: the product in int64 arithmetic, returned as complex128 (exact)."""
    ar, ai = a.real.astype(np.int64), a.imag.astype(np.int64)
    br, bi = b.real.astype(np.int64), b.imag.astype(np.int64)
    assert np.array_equal(ar, a.real) and np.array_equal(ai, a.imag) and np.array_equal(br, b.real) and np.array_equal(bi, b.imag)
    return (ar @ br - ai @ bi).astype(np.float64) + 1j * (ar @ bi + ai @ br).astype(np.float64)


def check_gemm_exact(c, a, b, what=""):
    ref = exact_product(a, b)
    bad = np.argwhere(~(c == ref))
    assert bad.size == 0, f"gemm exact {what}: {len(bad)} entries differ, first at {tuple(bad[0])}: {c[tuple(bad[0])]} vs {ref[tuple(bad[0])]}"


def check_gemm_accuracy(c, a, b, what=""):
    """elementwise bound against an extended-precision reference:  |C - AB| <= gamma (|Re A| + |Im A|)(|Re B| + |Im B|),
    gamma = 4 (k + 4) 2^-53.  The 3M form rounds (Re A + Im A)(Re B + Im B), so this, not |A||B|, is what it cancels against."""
    k = a.shape[1]
    ref = a.astype(np.clongdouble) @ b.astype(np.clongdouble)
    bound = 4.0 * (k + 4) * 2.0 ** -53 * ((np.abs(a.real) + np.abs(a.imag)) @ (np.abs(b.real) + np.abs(b.imag)))
    err = np.abs((c.astype(np.clongdouble) - ref)).astype(np.float64)
    ok = np.isfinite(c) & (err <= bound)
    bad = np.argwhere(~ok)
    assert bad.size == 0, f"gemm accuracy {what}: {len(bad)} entries out of bound, first at {tuple(bad[0])}: err {err[tuple(bad[0])]:.3e} > {bound[tuple(bad[0])]:.3e}"


# ---------------------------------------------------------------------------------------------------------------- SVD
SMALL_SMEM_MAX = 225 * 1024  # k_svd_small.cu: SMALL_SMEM_MAX
CL_C, CL_G, CL_MIN_P = 4, 8, 48   # k_svd_small.cu: cluster size, lanes per pair, smallest p of the cluster kernel
PAIRSUMS = 32                # kbp_jacobi.cuh: sizeof(PairSums)
TSVD_BMAX, TSVD_BMAX2, TSVD_B1 = 112, 192, 96   # k_tsvd.cu
CREG_BMAX = 96               # k_tsvd.cu: widest register-resident Cholesky
TSVD_PART_STRIDE = 160       # kbp_ops.cuh: keep <= 128 row sums of the check kernels + 2 norms


def svd_small_smem(m, n):
    """k_svd_small.cu: svd_small_smem"""
    p, q = min(m, n), (n if m <= n else m + n)
    return p * q * 16 + p * 12 + 16 + ((p + 1) // 2) * PAIRSUMS + 64


def svd_small_fits(m, n):
    """k_svd_small.cu: svd_small_fits"""
    return min(m, n) <= 128 and svd_small_smem(m, n) <= SMALL_SMEM_MAX


def small_kernel(m, n):
    """k_svd_small.cu: svd_small -- the kernel one launch of the in-shared-memory Jacobi SVD takes (a refused cluster launch,
    which the host code also handles, is not modelled)."""
    p = min(m, n)
    npairs = max((p + 1) // 2, 1)
    q = n if m <= n else m + n
    tall = m > n
    if p >= CL_MIN_P:
        cpl = cdiv(cdiv(q, CL_C), CL_G)
        if cpl <= 6 and npairs * CL_G <= 1024:
            return ("svd_cluster", cpl, CL_G, "tall" if tall else "wide")
    g = 32
    while g > 8 and npairs * g > 1024:
        g >>= 1
    threads = min(max(cdiv(npairs * g, 32) * 32, 256), 1024)
    cached = threads <= 768 and cdiv(q, g) <= 6
    return ("svd_small", cached, g)


def tsvd_block(m, n, keep):
    """k_tsvd.cu: tsvd_block (0: the subspace iteration does not apply)"""
    p = min(m, n)
    b = min(rup8(2 * keep), TSVD_BMAX2)
    if b < keep + 8 or b * 100 > p * 80:
        return 0
    return b


def chol_kernel(b):
    """k_tsvd.cu: launch_chol"""
    if b <= 32:
        return ("chol_reg", 1)
    if b <= 64:
        return ("chol_reg", 2)
    if b <= CREG_BMAX:
        return ("chol_reg", 3)
    return ("chol_blocked",)


def chol_blocks(b):
    """k_tsvd.cu: cholqr_pass -- one column block up to TSVD_BMAX, else 96 + the rest"""
    return [b] if b <= TSVD_BMAX else [TSVD_B1, b - TSVD_B1]


def svd_route(m, n, keep):
    """k_svd.cu: svd_truncate, svd_reducible; k_tsvd.cu: svd_truncate_subspace (keep > 128 -> exact path, it_max)."""
    p = min(m, n)
    if svd_small_fits(m, n):
        return {"route": "small", "kernel": small_kernel(m, n)}
    if p <= 128 and svd_small_fits(p, p):
        return {"route": "reduced", "kernel": small_kernel(p, p)}
    b = tsvd_block(m, n, keep)
    if b > 0 and keep <= 128:
        return {"route": "subspace", "b": b, "chol": [chol_kernel(x) for x in chol_blocks(b)], "rr": small_kernel(b, b),
                "it_max": 24 if 2 * b >= 5 * keep else 72}
    return {"route": "block_jacobi"}


def counter_delta(route, nb):
    """what one OP_SVD adds to Engine.svd_counters(): small / reduced are counted once per op by the host, the subspace
    and block-Jacobi decisions once per chain on the device (k_svd.cu, k_tsvd.cu: SvdCtl::counters)."""
    d = {"small": 0, "reduced": 0, "subspace": 0, "subspace_fallback": 0, "block_jacobi": 0}
    if route == "small":
        d["small"] = 1
    elif route == "reduced":
        d["reduced"] = 1
    elif route == "subspace":
        d["subspace"] = nb
    else:
        d["block_jacobi"] = nb
    return d


def subspace_shape(keep, kind):
    """m, n >= 1.25 b (+ 8), at least 136: square, tall or wide"""
    b = min(rup8(2 * keep), TSVD_BMAX2)
    p = max(rup8(cdiv(5 * b, 4)) + 8, 136)        # p > 128: neither the small kernel nor the Householder reduction takes it
    return {"square": (p, p), "tall": (p * 3 // 2, p), "wide": (p, p * 3 // 2)}[kind]


def subspace_decay(keep):
    """s_j = exp(-d j): the block resolves keep against b within a few iterations (factor exp(-2 d (b - keep)) per
    iteration) and the kept spectrum stays above the collapse test (s_keep / s_1 >= exp(-12) at 1.2 d)."""
    b = min(rup8(2 * keep), TSVD_BMAX2)
    return min(3.0 / (b - keep), 10.0 / keep)


SVD_KEEPS = [8, 16, 17, 32, 33, 48, 49, 56, 57, 64, 65, 80, 81, 96, 100, 128]
SVD_KEEP_EXACT = 129

# small / reduced / exact variants: name -> (m, n, keep)
SVD_SMALL = {
    "40x100": (40, 100, 12),
    "20x600": (20, 600, 8), "600x20": (600, 20, 8),
    "65x200": (65, 200, 20), "130x65": (130, 65, 20),
    "48x60": (48, 60, 16), "50x90": (50, 90, 16), "60x120": (60, 120, 20), "64x150": (64, 150, 20), "81x162": (81, 162, 18),
    "60x48": (60, 48, 16), "100x50": (100, 50, 16), "130x60": (130, 60, 20),
    "32x449": (32, 449, 10), "417x32": (417, 32, 10),        # just past the small kernel's shared memory: reduced
    "128x600": (128, 600, 32), "600x128": (600, 128, 32),    # subspace
    "200x160": (200, 160, 150),                              # block-Jacobi
}
SVD_SMALL_EXPECT = {
    "40x100": ("small", ("svd_small", True, 32)),
    "20x600": ("small", ("svd_small", False, 32)), "600x20": ("small", ("svd_small", False, 32)),
    "65x200": ("small", ("svd_small", False, 16)), "130x65": ("small", ("svd_small", False, 16)),
    "48x60": ("small", ("svd_cluster", 2, 8, "wide")), "50x90": ("small", ("svd_cluster", 3, 8, "wide")),
    "60x120": ("small", ("svd_cluster", 4, 8, "wide")), "64x150": ("small", ("svd_cluster", 5, 8, "wide")),
    "81x162": ("small", ("svd_cluster", 6, 8, "wide")),
    "60x48": ("small", ("svd_cluster", 4, 8, "tall")), "100x50": ("small", ("svd_cluster", 5, 8, "tall")),
    "130x60": ("small", ("svd_cluster", 6, 8, "tall")),
    "32x449": ("reduced", ("svd_small", True, 32)), "417x32": ("reduced", ("svd_small", True, 32)),
    "128x600": ("subspace", None), "600x128": ("subspace", None),
    "200x160": ("block_jacobi", None),
}

# one representative per route for the hard inputs: name -> (m, n, keep)
SVD_HARD_ROUTES = {"small": (40, 100, 12), "small_streamed": (20, 600, 8), "cluster_wide": (60, 120, 20),
                   "cluster_tall": (100, 50, 16), "reduced": (417, 32, 10), "subspace": (300, 260, 24),
                   "subspace_wide": (272, 272, 60), "block_jacobi": (200, 160, 150)}
SVD_HARD_INPUTS = ["repeated_at_cut", "flat", "rank_below_keep", "rank_between_keep_and_b", "zero", "tiny_rows"]


def _haar(rng, n, k):
    q, r = np.linalg.qr(rng.normal(size=(n, k)) + 1j * rng.normal(size=(n, k)))
    return q * (np.diag(r) / np.abs(np.diag(r)))


def with_spectrum(rng, m, n, s):
    p = min(m, n)
    s = np.asarray(s, dtype=np.float64)
    return (_haar(rng, m, p) * s) @ _haar(rng, n, p).conj().T


def hard_input(rng, kind, m, n, keep):
    """the hard inputs of the SVD routes"""
    p = min(m, n)
    b = min(rup8(2 * keep), TSVD_BMAX2)
    if kind == "repeated_at_cut":          # exactly equal singular values from keep - 2 to keep + 2 (4 on each side when room)
        s = np.exp(-0.1 * np.arange(p))
        lo, hi = max(keep - 3, 0), min(keep + 3, p)
        s[lo:hi] = s[lo]
        return with_spectrum(rng, m, n, np.sort(s)[::-1])
    if kind == "flat":
        return with_spectrum(rng, m, n, np.full(p, 1.7))
    if kind == "rank_below_keep":
        r = max(keep // 2, 1)
        return with_spectrum(rng, m, n, np.where(np.arange(p) < r, np.exp(-0.2 * np.arange(p)), 0.0))
    if kind == "rank_between_keep_and_b":
        r = min(max(keep + 2, (keep + b) // 2), p)
        return with_spectrum(rng, m, n, np.where(np.arange(p) < r, np.exp(-0.2 * np.arange(p)), 0.0))
    if kind == "zero":
        return np.zeros((m, n), complex)
    if kind == "tiny_rows":                # an O(1) matrix with a decaying spectrum, half its rows scaled to 1e-150
        a = with_spectrum(rng, m, n, np.exp(-0.15 * np.arange(p)))
        a[m // 2:] *= 1e-150
        return a
    raise ValueError(kind)


class SvdCheckError(AssertionError):
    pass


def check_svd(a, us, vh, slots, keep, nr_bulk, slot_lognorm=0, slot_trunc=1, what=""):
    """gap-free check of a rank-`keep` truncated SVD US Vh (US scaled by 1 / ||A||_F when nr_bulk) against float64 LAPACK:
    Eckart-Young error, column norms of US = the leading singular values, orthonormal rows of Vh where s_j > 1e-10 s_1,
    the lognorm / truncation / status slots, no non-finite entries.  Raises SvdCheckError naming the failed check."""
    def need(cond, name, detail=""):
        if not cond:
            raise SvdCheckError(f"svd {what}: {name} {detail}")
    need(np.all(np.isfinite(us)) and np.all(np.isfinite(vh)), "non-finite output")
    s = np.linalg.svd(a, compute_uv=False)
    fro = float(np.linalg.norm(s))
    f = fro if (nr_bulk and fro > 0) else 1.0
    err = float(np.linalg.norm(a - (us * f) @ vh))
    tail = float(np.sqrt(np.sum(s[keep:] ** 2)))
    need(err <= tail + 1e-12 * fro, "Eckart-Young", f"err {err:.6e} > tail {tail:.6e} + 1e-12 |A| ({fro:.3e})")
    cn = np.linalg.norm(us, axis=0) * f
    need(np.allclose(np.sort(cn)[::-1], s[:keep], rtol=1e-10, atol=1e-12 * (s[0] if fro > 0 else 0.0)), "column norms",
         f"{np.max(np.abs(np.sort(cn)[::-1] - s[:keep])):.3e}")
    big = cn > 1e-10 * (s[0] if fro > 0 else 0.0)
    if big.any():
        g = (vh[big] @ vh[big].conj().T)
        need(np.linalg.norm(g - np.eye(int(big.sum()))) <= 1e-10, "Vh orthonormal", f"{np.linalg.norm(g - np.eye(int(big.sum()))):.3e}")
    terr = float(np.sqrt(np.sum(s[keep:] ** 2) / np.sum(s ** 2))) if fro > 0 else 0.0
    need(abs(slots[slot_trunc] - terr) <= 1e-10, "truncation slot", f"{slots[slot_trunc]} vs {terr}")
    ln = np.log(fro) if (nr_bulk and fro > 0) else 0.0
    need(abs(slots[slot_lognorm] - ln) <= 1e-12 * max(1.0, abs(ln)), "lognorm slot", f"{slots[slot_lognorm]} vs {ln}")
    need(slots[-1] == 0, "status slot", f"{slots[-1]}")


# ---------------------------------------------------------------------------------------------------------------- QR
QRC_MLOC_MAX, QRC_SMEM_MAX = 128, 220 * 1024   # k_qr_cluster.cu


def qr_route(m, n):
    """k_qr.cu: qr; k_tsvd.cu: qr_cholqr2 (8 <= n <= 96, m >= 4 n, workspace), qr_blocked (m >= n >= 128, workspace)."""
    k = min(m, n)
    nblk = cdiv(n, 16)
    if 8 <= n <= CREG_BMAX and m >= 4 * n and m * n + 4 * n * n + 2 * n * n + n + nblk * 256 + 8 <= m * n + m * k + k + 8:
        return "cholqr2"
    if m >= n >= 128:
        nblocks = cdiv(n, 64)
        w = rup8(cdiv(n, nblocks))
        need = (n * m + 2 * m * w + 2 * n * w + w * w) + (2 * m * w + w + 8)
        if need <= 2 * m * n + n + 8:
            return "blocked"
    return "householder"


# extra QR shapes (test_kernels_gpu.py::test_qr): one per route edge
QR_CASES = {(208, 32): "cholqr2", (207, 32): "householder", (592, 96): "cholqr2", (584, 96): "householder",
            (600, 97): "householder", (392, 392): "blocked", (384, 384): "householder", (816, 264): "blocked",
            (300, 8): "cholqr2", (300, 7): "householder", (32, 96): "householder"}


# ---------------------------------------------------------------------------------------------------------------- table
def gemm_instantiations():
    return {("zgemm", t, akc, bkc) for t in (16, 32, 64) for akc in (True, False) for bkc in (True, False)}


INSTANTIATIONS = (gemm_instantiations()
                  | {("svd_small", True, 32), ("svd_small", False, 32), ("svd_small", False, 16)}
                  | {("svd_cluster", c, 8, mode) for c in range(2, 7) for mode in ("wide",)}
                  | {("svd_cluster", c, 8, "tall") for c in (4, 5, 6)}
                  | {("chol_reg", 1), ("chol_reg", 2), ("chol_reg", 3), ("chol_blocked",)})
UNREACHABLE = {("svd_small", True, 8), ("svd_small", False, 8), ("svd_small", True, 16), ("svd_cluster", 1, 8, "wide"),
               ("svd_cluster", 1, 8, "tall")}


def reached_instantiations():
    """every kernel instantiation the case tables reach, by the mirror"""
    got = set()
    for m, n, k, nb in list(GEMM_CASES.values()) + list(GEMM_POISON.values()):
        for oa in range(4):
            for ob in range(4):
                got.add(gemm_kernel(m, n, k, nb, oa, ob))
    for m, n, keep in SVD_SMALL.values():
        r = svd_route(m, n, keep)
        if "kernel" in r:
            got.add(r["kernel"])
    for keep in SVD_KEEPS:
        for kind in ("square", "tall", "wide"):
            m, n = subspace_shape(keep, kind)
            r = svd_route(m, n, keep)
            if r["route"] == "subspace":
                got.update(r["chol"])
                got.add(r["rr"])
    return got
