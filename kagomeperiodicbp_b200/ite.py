"""Two-site reduced density matrix and full-update gate application on an edge with a periodic-MPS environment -- the
S4 seam of the reference (src/libs/ITE.py):

    rho_ij(Ti, Tj, mps_env=...)                       ITE.py:555-761   (mps_env branch :683-756)
    reduced_env(Ti, Tj, mps_env=...)                  ITE.py:853-1302
    reduced_inner_prod / truncation_distance          ITE.py:1309-1355
    Ni_env / Nj_env / robust_solve                    ITE.py:1394-1509
    ALS_optimization                                  ITE.py:1518-1753
    apply_2local_gate(g, Dmax, Ti, Tj, mps_env=...)   ITE.py:1761-2020
    g_from_exp_h                                      ITE.py:2027-2068

Conventions are the reference's: Ti = [d, D_shared, k1, k2, k3], mps_env = six tensors [D_L, D, D*, D_R] that start at the
first non-shared leg of Ti and run counter-clockwise around the pair.

Every dense operation goes through a backend object ``B`` (``linalg.DeviceBackend`` in the product: each tensordot / QR /
SVD / eigh is a device program run through the C ABI; there is no CPU fallback).  Host code only moves data (reshape,
transpose, slicing) and takes scalar decisions on eigen/singular values (how many to keep, whether to regularise), as the
reference does in Python.

Differences from the reference that do not change any result:
  * numpy.linalg.solve on the (Hermitian, positive semi-definite) ALS normal matrices is an eigen-decomposition solve here;
    the regularisation rule of robust_solve (|x| > 1e8 |b| / |N|  ->  N + 1e-8 |N|_2) is kept.
  * QR / SVD / eigh gauges differ (Householder and Jacobi kernels instead of LAPACK); everything returned is compared through
    gauge-invariant quantities (RDM, energies, N_red spectrum, the pair tensor contracted over its bond).
"""
from __future__ import annotations

import numpy as np

PINV_THRESH = 1e-8         # ITE.py:98
ROBUST_THRESH = 1e8        # ITE.py:99
TRUNC_POS_EPS = 1e-12      # ITE.py:1205


class ITEError(RuntimeError):
    """(src/_error_types.py) raised e.g. when N_red has no positive eigenvalue (ITE.py:1200-1201)."""


def _half_env(B, T, envs):
    """contract a site tensor T[p, s, k1..kn] and its conjugate with its n environment tensors [L, k, k*, R]:
    returns [p, p*, s, s*, L_first, R_last]."""
    n = T.ndim - 2
    X = B.tensordot(T, envs[0], ([2], [1]))                          # [p, s, k2.., L, b1, R]
    nd = X.ndim
    X = B.transpose(X, [0, 1, nd - 3] + list(range(2, nd - 3)) + [nd - 2, nd - 1])   # [p, s, L, k2.., b1, R]
    for e in envs[1:n]:
        X = B.tensordot(X, e, ([3, X.ndim - 1], [1, 0]))             # [p, s, L, k.., b.., R]
    # X = [p, s, L, b1..bn, R]
    X = B.tensordot(X, T, (list(range(3, 3 + n)), list(range(2, 2 + n))), conj_b=True)   # [p, s, L, R, p*, s*]
    return B.transpose(X, [0, 4, 1, 5, 2, 3])


def rho_ij_unnormalized(B, Ti, Tj, mps_env):
    """the contraction of ``rho_ij`` without its trace normalisation: rho[i, i*, j, j*] as a tensor of the backend ``B``.
    Only backend operations, no host value: a compiled program can record it."""
    ni = Ti.ndim - 2
    Ai = _half_env(B, Ti, mps_env[:ni])                              # [p, p*, s, s*, L0, R_last]
    Aj = _half_env(B, Tj, mps_env[ni:])
    # ring closure: left bond of env_i[0] with right bond of env_j[-1], right bond of env_i[-1] with left bond of env_j[0]
    return B.tensordot(Ai, Aj, ([2, 3, 4, 5], [2, 3, 5, 4]))


def rho_trace(rho) -> complex:
    """trace of a two-site RDM rho[i, i*, j, j*] (a d^4 host reduction)."""
    return np.trace(np.trace(np.asarray(rho), axis1=0, axis2=1))


def rho_ij(B, Ti, Tj, mps_env):
    """(ITE.py:683-756)  rho[i, i*, j, j*], trace normalised."""
    rho = rho_ij_unnormalized(B, Ti, Tj, mps_env)
    return np.asarray(B.scale(rho, 1.0 / rho_trace(rho)))


def _n_half(B, T_rest, envs, n_legs):
    """N_i[Dred, Dred*, L, R] of ITE.py:1046-1096 (T_rest = [Dred, k1..kn])."""
    N_ = B.tensordot(T_rest, envs[0], ([1], [1]))                    # [Dred, k2.., L, b1, R]
    l = N_.ndim
    N_ = B.transpose(N_, [0, l - 3] + list(range(1, l - 3)) + [l - 2, l - 1])        # [Dred, L, k2.., b1, R]
    for mp in envs[1:n_legs]:
        N_ = B.tensordot(N_, mp, ([2, N_.ndim - 1], [1, 0]))
    N_ = B.tensordot(N_, T_rest, (list(range(2, 2 + n_legs)), list(range(1, 1 + n_legs))), conj_b=True)   # [Dred, L, R, Dred*]
    return N_


def _pinv(B, M, rcond):
    """numpy.linalg.pinv(M, rcond) from a device SVD."""
    U, S, Vh = B.svd(M)
    keep = S > rcond * (S[0] if len(S) else 0.0)
    w = np.where(keep, 1.0 / np.where(keep, S, 1.0), 0.0)
    VS = B.tensordot(Vh, np.diag(w).astype(np.complex128), ([0], [0]), conj_a=True)      # V diag(w)   [n, k]
    return B.tensordot(VS, U, ([1], [1]), conj_b=True)                                       # V diag(w) U^H


def rho_from_reduced(N4, ai, aj):
    """the two-site RDM from the REDUCED environment: with T_i = a_i T_i_rest, T_j = a_j T_j_rest and
    N4[a, a*, b, b*] = (environment ring contracted with T_i_rest, T_j_rest and their conjugates),
        rho[p, p*, q, q*] = sum  a_i[p, s, a] conj(a_i[p*, s*, a*])  a_j[q, s, b] conj(a_j[q*, s*, b*])  N4[a, a*, b, b*]
    is the same contraction as ``rho_ij`` (ITE.py:683-756) in another order -- (d D)^4 numbers on the host instead of a second and
    third pass over the chi D^2-bond ring tensors (the dominant cost of ``rho_ij``).  Trace normalised."""
    N4, ai, aj = np.asarray(N4), np.asarray(ai), np.asarray(aj)
    ket = np.tensordot(ai, aj, ([1], [1]))                                   # [p, a, q, b]
    t = np.tensordot(ket, N4, ([1, 3], [0, 2]))                              # [p, q, a*, b*]
    bra = np.conj(ket)                                                       # [p*, a*, q*, b*]
    rho = np.tensordot(t, bra, ([2, 3], [1, 3]))                             # [p, q, p*, q*]
    rho = rho.transpose(0, 2, 1, 3)
    tr = np.trace(np.trace(rho, axis1=0, axis2=1))
    return rho / tr


def reduced_env(B, Ti, Tj, mps_env, aux=None):
    """(ITE.py:853-1302, mps_env branch)  -> X[Di, Dj, DX], ai[d, D, Di], aj[d, D, Dj], Ti_rest, Tj_rest, w (spectrum of N_red).
    ``aux`` (dict, optional): receives what ``rho_from_reduced`` needs -- N4 (the environment on the reduced legs, before it is
    hermitised), the factors a_i, a_j of the ORIGINAL tensors and the two gauge matrices applied to the rest tensors."""
    d, D = Ti.shape[0], Ti.shape[1]
    Di_rest, Dj_rest = Ti.size // (d * D), Tj.size // (d * D)
    n_i, n_j = Ti.ndim - 2, Tj.ndim - 2
    # Ti_mat^T = Q R  ->  Ti_rest = Q^T [Dred, rest],  ai = R^T [d D, Dred]
    Q, R = B.qr(B.transpose(B.reshape(Ti, (d * D, Di_rest)), (1, 0)))
    Ti_rest, ai = B.transpose(Q, (1, 0)), B.transpose(R, (1, 0))
    Di_red = ai.shape[1]
    ai = B.reshape(ai, (d, D, Di_red))
    Q, R = B.qr(B.transpose(B.reshape(Tj, (d * D, Dj_rest)), (1, 0)))
    Tj_rest, aj = B.transpose(Q, (1, 0)), B.transpose(R, (1, 0))
    Dj_red = aj.shape[1]
    aj = B.reshape(aj, (d, D, Dj_red))

    Ti_rest = B.reshape(Ti_rest, (Di_red,) + tuple(Ti.shape[2:]))
    Ni = B.transpose(_n_half(B, Ti_rest, mps_env[:n_i], n_i), (0, 3, 1, 2))            # [Dred, Dred*, L(up), R(down)]
    Tj_rest = B.reshape(Tj_rest, (Dj_red,) + tuple(Tj.shape[2:]))
    Nj = B.transpose(_n_half(B, Tj_rest, mps_env[n_i:], n_j), (0, 3, 2, 1))            # [Dred, Dred*, R(up), L(down)]
    Ti_rest = B.reshape(Ti_rest, (Di_red, Ti_rest.size // Di_red))
    Tj_rest = B.reshape(Tj_rest, (Dj_red, Tj_rest.size // Dj_red))
    Ni = B.scale(Ni, 1.0 / B.norm(Ni))
    Nj = B.scale(Nj, 1.0 / B.norm(Nj))
    Nred = B.tensordot(Ni, Nj, ([2, 3], [2, 3]))                                       # [Di, Di*, Dj, Dj*]
    if aux is not None:
        aux.update(N4=np.asarray(Nred).copy(), ai0=np.asarray(ai).copy(), aj0=np.asarray(aj).copy())
    Nred = B.reshape(B.transpose(Nred, (0, 2, 1, 3)), (Di_red * Dj_red, Di_red * Dj_red))
    Nred = B.hermitize(Nred)
    w, U = B.eigh(Nred)                                                                # ascending
    if np.all(w < 0):
        raise ITEError("No positive eigen-values!")
    pos = int(np.where(w > TRUNC_POS_EPS * w[-1])[0][0])
    wpos = w[pos:]
    X = B.tensordot(U[:, pos:], np.diag(np.sqrt(wpos)).astype(np.complex128), ([1], [0]))
    DX = X.shape[1]
    X = B.reshape(X, (Di_red, Dj_red, DX))
    # gauge fixing of the two reduced legs (ITE.py:1239-1285)
    _, Ri = B.qr(B.transpose(B.reshape(X, (Di_red, Dj_red * DX)), (1, 0)))
    Li = B.transpose(Ri, (1, 0))
    Li_inv = _pinv(B, Li, PINV_THRESH)
    Xt = B.reshape(B.transpose(X, (0, 2, 1)), (Di_red * DX, Dj_red))
    _, Rj = B.qr(Xt)
    Rj_inv = _pinv(B, Rj, PINV_THRESH)
    X = B.tensordot(Li_inv, X, ([1], [0]))
    Ti_rest = B.tensordot(Li_inv, Ti_rest, ([1], [0]))
    ai = B.tensordot(ai, Li, ([2], [0]))
    X = B.transpose(B.tensordot(X, Rj_inv, ([1], [0])), (0, 2, 1))
    Tj_rest = B.transpose(B.tensordot(Tj_rest, Rj_inv, ([0], [0])), (1, 0))
    aj = B.tensordot(aj, Rj, ([2], [1]))
    if aux is not None:
        aux.update(Li_inv=np.asarray(Li_inv).copy(), Rj_inv=np.asarray(Rj_inv).copy())
    Di_red, Dj_red = ai.shape[2], aj.shape[2]
    Ti_rest = B.reshape(Ti_rest, (Di_red,) + tuple(Ti.shape[2:]))
    Tj_rest = B.reshape(Tj_rest, (Dj_red,) + tuple(Tj.shape[2:]))
    return X, ai, aj, Ti_rest, Tj_rest, w


def reduced_inner_prod(B, ai_ket, aj_ket, ai_bra, aj_bra, X):
    """(ITE.py:1309-1331)"""
    ket = B.tensordot(ai_ket, X, ([2], [0]))
    ket = B.tensordot(aj_ket, ket, ([1, 2], [1, 2]))
    bra = B.tensordot(ai_bra, X, ([2], [0]))
    bra = B.tensordot(aj_bra, bra, ([1, 2], [1, 2]))
    return complex(np.asarray(B.tensordot(ket, bra, ([0, 1, 2], [0, 1, 2]), conj_b=True)).reshape(-1)[0])


def truncation_distance(B, exact_ai, exact_aj, new_ai, new_aj, X):
    """(ITE.py:1334-1355)"""
    ip1 = reduced_inner_prod(B, exact_ai, exact_aj, exact_ai, exact_aj, X)
    ip2 = reduced_inner_prod(B, new_ai, new_aj, new_ai, new_aj, X)
    ip3 = reduced_inner_prod(B, exact_ai, exact_aj, new_ai, new_aj, X)
    return float((2 * (ip1 + ip2 - 2 * ip3) / (ip1 + ip2)).real)


def Ni_env(B, aj_ket, aj_bra, X):
    """(ITE.py:1394-1429)  -> [d, D, Dred(i); d*, D*, Dred(i)*]"""
    d = aj_ket.shape[0]
    ket = B.tensordot(aj_ket, X, ([2], [1]))                          # [d, D, Dred(i), DX]
    bra = B.tensordot(aj_bra, X, ([2], [1]))
    N_ = B.tensordot(ket, bra, ([0, 3], [0, 3]), conj_b=True)         # [D, Dred(i), D*, Dred(i)*]
    N_ = B.tensordot(np.eye(d, dtype=np.complex128), N_, 0)
    return B.transpose(N_, (0, 2, 3, 1, 4, 5))


def Nj_env(B, ai_ket, ai_bra, X):
    """(ITE.py:1432-1449)"""
    return Ni_env(B, ai_ket, ai_bra, B.transpose(X, (1, 0, 2)))


def robust_solve(B, N_, b):
    """(ITE.py:1452-1509) for a Hermitian positive semi-definite N: x = V diag(1 / lam) V^H b, regularised like the
    reference when the plain solve blows up."""
    w, V = B.eigh(B.hermitize(N_))
    nN = float(np.sqrt(np.sum(w ** 2)))                                # Frobenius norm of a Hermitian matrix
    nb = B.norm(b)
    Vb = B.tensordot(V, np.asarray(b).reshape(-1, 1), ([0], [0]), conj_a=True)          # V^H b
    regularize = bool(np.any(w == 0.0))
    x = None
    if not regularize:
        x = B.tensordot(V, B.tensordot(np.diag(1.0 / w).astype(np.complex128), Vb, ([1], [0])), ([1], [0]))
        nx = B.norm(x)
        if not np.isfinite(nx) or nx > ROBUST_THRESH * nb / nN:
            regularize = True
    if regularize:
        shift = PINV_THRESH * float(np.max(np.abs(w)))                 # |N|_2 of a Hermitian matrix
        x = B.tensordot(V, B.tensordot(np.diag(1.0 / (w + shift)).astype(np.complex128), Vb, ([1], [0])), ([1], [0]))
    return B.reshape(x, (-1,))


def ALS_optimization(B, Dmax, exact_ai, exact_aj, X, iter_max=10, eps=1e-6):
    """(ITE.py:1518-1753)"""
    D = exact_ai.shape[1]
    if D <= Dmax:
        return exact_ai.copy(), exact_aj.copy()
    new_ai = np.ascontiguousarray(exact_ai[:, 0:Dmax, :])
    new_aj = np.ascontiguousarray(exact_aj[:, 0:Dmax, :])
    iter_no, dist, delta = 0, 1e10, 1.0
    while delta > eps and iter_no < iter_max:
        Ni = Ni_env(B, new_aj, new_aj, X)
        s = Ni.shape
        Ni = B.transpose(B.reshape(Ni, (s[0] * s[1] * s[2], s[3] * s[4] * s[5])), (1, 0))
        Nib = Ni_env(B, exact_aj, new_aj, X)
        b = B.reshape(B.tensordot(Nib, exact_ai, ([0, 1, 2], [0, 1, 2])), (-1,))
        new_ai = B.reshape(robust_solve(B, Ni, b), new_ai.shape)
        Nj = Nj_env(B, new_ai, new_ai, X)
        s = Nj.shape
        Nj = B.transpose(B.reshape(Nj, (s[0] * s[1] * s[2], s[3] * s[4] * s[5])), (1, 0))
        Njb = Nj_env(B, exact_ai, new_ai, X)
        b = B.reshape(B.tensordot(Njb, exact_aj, ([0, 1, 2], [0, 1, 2])), (-1,))
        new_aj = B.reshape(robust_solve(B, Nj, b), new_aj.shape)
        # balance the bond (ITE.py:1700-1731)
        ai = B.transpose(new_ai, (0, 2, 1))
        ai_shape = ai.shape
        Qi, Ri = B.qr(B.reshape(ai, (ai_shape[0] * ai_shape[1], ai_shape[2])))
        aj = B.transpose(new_aj, (1, 0, 2))
        aj_shape = aj.shape
        Qj, Rj = B.qr(B.transpose(B.reshape(aj, (aj_shape[0], aj_shape[1] * aj_shape[2])), (1, 0)))
        Qj, Lj = B.transpose(Qj, (1, 0)), B.transpose(Rj, (1, 0))
        U, S, V = B.svd(B.tensordot(Ri, Lj, ([1], [0])))
        sq = np.diag(np.sqrt(S)).astype(np.complex128)
        Qi = B.tensordot(B.tensordot(Qi, U, ([1], [0])), sq, ([1], [0]))
        Qj = B.tensordot(B.tensordot(sq, V, ([1], [0])), Qj, ([1], [0]))
        new_ai = B.transpose(B.reshape(Qi, ai_shape), (0, 2, 1))
        new_aj = B.transpose(B.reshape(Qj, aj_shape), (1, 0, 2))
        old = dist
        dist = truncation_distance(B, exact_ai, exact_aj, new_ai, new_aj, X)
        delta = abs(dist - old)
        iter_no += 1
    new_ai = B.scale(new_ai, 1.0 / B.norm(new_ai))
    new_aj = B.scale(new_aj, 1.0 / B.norm(new_aj))
    ALS_optimization.last = dict(iterations=iter_no, distance=dist)
    return new_ai, new_aj


def apply_2local_gate(B, g, Dmax, Ti, Tj, mps_env, aux=None):
    """(ITE.py:1761-2020)  -> (Ti_new, Tj_new, spectrum of N_red | None).
    ``aux`` (dict, optional, not in the reference): when the gate goes through the reduced environment it receives
    ``rho_before`` and ``rho_after``, the two-site RDMs of (Ti, Tj) and of (Ti_new, Tj_new) in this environment computed from
    the reduced environment (``rho_from_reduced``) -- what the update loop would otherwise get from two more ``rho_ij`` calls."""
    g = np.asarray(g, dtype=np.complex128)
    gm = g.transpose(0, 2, 1, 3).reshape(g.shape[0] * g.shape[2], g.shape[1] * g.shape[3])
    sc = np.linalg.norm(gm, ord=2)                                    # 4 x 4 host scalar checks, as in the reference
    if sc < 1e-15:
        raise ITEError("apply_2local_gate: the gate vanishes")
    if np.linalg.norm(gm - gm[0, 0] * np.eye(gm.shape[0])) / sc < 1e-10:
        return Ti, Tj, None
    s = np.linalg.svd(g.reshape(g.shape[0] * g.shape[1], g.shape[2] * g.shape[3]), compute_uv=False)
    if s.shape[0] == 0 or s[1] / s[0] < 1e-10:                        # product gate: no truncation needed (ITE.py:1893-1930)
        mi = np.unravel_index(np.abs(g).argmax(), g.shape)
        g_i, g_j = g[:, :, mi[2], mi[3]], g[mi[0], mi[1], :, :]
        rescale = g[mi] / (g_i[mi[0], mi[1]] * g_j[mi[2], mi[2]])
        fi = np.sqrt(abs(rescale))
        return (np.asarray(B.tensordot(fi * g_i, Ti, ([1], [0]))), np.asarray(B.tensordot((rescale / fi) * g_j, Tj, ([1], [0]))), None)
    red = {} if aux is not None else None
    X, ai, aj, Ti_rest, Tj_rest, w = reduced_env(B, Ti, Tj, mps_env, aux=red)
    d, Di_red, Dj_red = ai.shape[0], ai.shape[2], aj.shape[2]
    ex = B.tensordot(ai, aj, ([1], [1]))                               # [d, Di, d, Dj]
    ex = B.tensordot(g, ex, ([1, 3], [0, 2]))                          # [d, d, Di, Dj]
    ex = B.reshape(B.transpose(ex, (0, 2, 1, 3)), (d * Di_red, d * Dj_red))
    U, S, V = B.svd(ex)
    sq = np.diag(np.sqrt(S)).astype(np.complex128)
    exact_ai = B.tensordot(U, sq, ([1], [0]))
    exact_aj = B.tensordot(sq, V, ([1], [0]))
    Dp = exact_ai.shape[1]
    exact_ai = B.transpose(B.reshape(exact_ai, (d, Di_red, Dp)), (0, 2, 1))
    exact_aj = B.transpose(B.reshape(exact_aj, (Dp, d, Dj_red)), (1, 0, 2))
    new_ai, new_aj = ALS_optimization(B, Dmax, exact_ai, exact_aj, X)
    if aux is not None:
        # T_i_new = new_ai (Li_inv T_i_rest0), T_j_new = new_aj (T_j_rest0 Rj_inv): the factors on the ORIGINAL rest tensors
        ai_eff = np.tensordot(np.asarray(new_ai), red["Li_inv"], ([2], [0]))
        aj_eff = np.tensordot(np.asarray(new_aj), red["Rj_inv"], ([2], [1]))
        aux["rho_before"] = rho_from_reduced(red["N4"], red["ai0"], red["aj0"])
        aux["rho_after"] = rho_from_reduced(red["N4"], ai_eff, aj_eff)
    new_Ti = B.tensordot(new_ai, Ti_rest, ([2], [0]))
    new_Tj = B.tensordot(new_aj, Tj_rest, ([2], [0]))
    new_Ti = np.asarray(B.scale(new_Ti, 1.0 / float(np.max(np.abs(np.asarray(new_Ti))))))
    new_Tj = np.asarray(B.scale(new_Tj, 1.0 / float(np.max(np.abs(np.asarray(new_Tj))))))
    return new_Ti, new_Tj, w


def g_from_exp_h(h, dt):
    """(ITE.py:2027-2068)  4 x 4 host matrix exponential, as the reference (scipy.linalg.expm)."""
    from scipy.linalg import expm
    d = h.shape[0]
    hm = np.asarray(h).transpose(0, 2, 1, 3).reshape(d * d, d * d)
    return expm(-dt * hm).reshape(d, d, d, d).transpose(0, 2, 1, 3)


def heisenberg_afm():
    """(src/physics/hamiltonians.py:53-57)  h[i, i*, j, j*] = Sx Sx + Sy Sy + Sz Sz."""
    sx = np.array([[0, 1], [1, 0]], dtype=np.complex128) / 2
    sy = np.array([[0, -1j], [1j, 0]], dtype=np.complex128) / 2
    sz = np.array([[1, 0], [0, -1]], dtype=np.complex128) / 2
    return sum(np.tensordot(s, s, 0) for s in (sx, sy, sz))
