"""TEST INFRASTRUCTURE (CPU oracle) -- a plain numpy statement of the simple update (Jiang, Weng and Xiang, PRL 101, 090603
(2008)) of the three-site Kagome unit cell on the Gamma / lambda representation, written without the package's code.  Only
tests/ and tools/ may import this module.

State: gammas = [Gamma_A, Gamma_B, Gamma_C], each [d, D, D, D, D] (leg order of UnitCell), and lams = six positive vectors of
length D, one per bond.  ``table`` lists the bonds as (site_i, leg_i, site_j, leg_j) with virtual leg indices 0..3; one SU
step updates them in table order (first-order Trotter).  One bond update:

  1. T = Gamma with the lambdas of its three other legs absorbed, for both sites
  2. M = T reshaped to [D^3 (other legs, in leg order), d * D (physical, bond)], M = Q R
  3. theta[a, p', b, q'] = sum g[p', p, q', q] R_i[a, p, k] lambda_b[k] R_j[b, q, k]      (g in ite.g_from_exp_h's layout)
  4. SVD of theta as (d r_i) x (d r_j), keep D
  5. lambda_b = S[:D] / |S[:D]|
  6. Gamma_i = Q_i U, Gamma_j = Q_j conj(V), the other legs' lambdas divided back out (entries below LAMBDA_CUTOFF * max
     get a zero inverse)
  7. Gamma_i, Gamma_j scaled to unit Frobenius norm

A step's convergence measure is max over bonds of |lambda_b(new) - lambda_b(old)|_2.
"""
from __future__ import annotations

import numpy as np

LAMBDA_CUTOFF = 1e-12


def leg_bonds(table):
    """legb[site][leg] = index of the bond that leg belongs to."""
    legb = [[None] * 4 for _ in range(3)]
    for b, (i, li, j, lj) in enumerate(table):
        legb[i][li] = b
        legb[j][lj] = b
    return legb


def _inv(lam):
    lam = np.asarray(lam, dtype=np.float64)
    cut = LAMBDA_CUTOFF * np.max(lam) if lam.size else 0.0
    return np.where(lam > cut, 1.0 / np.where(lam > cut, lam, 1.0), 0.0)


def _scale_leg(T, leg, v):
    """multiply virtual leg ``leg`` (0..3) of T[p, l0, l1, l2, l3] by the vector v."""
    shape = [1] * 5
    shape[leg + 1] = v.size
    return T * v.reshape(shape)


def _with_outer(G, site, skip, lams, legb, power=1.0):
    T = G
    for l in range(4):
        if l != skip:
            T = _scale_leg(T, l, np.asarray(lams[legb[site][l]], dtype=np.float64) ** power)
    return T


def _to_matrix(T, leg):
    """[p, l0..l3] -> [(other legs), (p, leg)]"""
    others = [l + 1 for l in range(4) if l != leg]
    d, D = T.shape[0], T.shape[1]
    return T.transpose(others + [0, leg + 1]).reshape(D ** 3, d * D)


def _from_matrix(M, leg, d, D):
    """inverse of _to_matrix"""
    others = [l + 1 for l in range(4) if l != leg]
    order = others + [0, leg + 1]
    inv = np.argsort(order)
    return M.reshape(D, D, D, d, D).transpose(inv)


def bond_update(gammas, lams, b, g, table):
    """one bond update; returns new (gammas, lams) lists (inputs untouched)."""
    gammas, lams = list(gammas), [np.asarray(l, dtype=np.float64).copy() for l in lams]
    legb = leg_bonds(table)
    i, li, j, lj = table[b]
    d, D = gammas[i].shape[0], gammas[i].shape[1]
    Qi, Ri = np.linalg.qr(_to_matrix(_with_outer(gammas[i], i, li, lams, legb), li))
    Qj, Rj = np.linalg.qr(_to_matrix(_with_outer(gammas[j], j, lj, lams, legb), lj))
    r_i, r_j = Ri.shape[0], Rj.shape[0]
    theta = np.einsum("apk,k,bqk->apbq", Ri.reshape(r_i, d, D), lams[b], Rj.reshape(r_j, d, D))
    theta = np.einsum("PpQq,apbq->aPbQ", np.asarray(g), theta)
    U, S, Vh = np.linalg.svd(theta.reshape(r_i * d, r_j * d))
    U, S, Vh = U[:, :D], S[:D], Vh[:D]
    lams[b] = S / np.linalg.norm(S)
    for site, leg, Q, Y, r in ((i, li, Qi, U, r_i), (j, lj, Qj, Vh.T, r_j)):
        G = _from_matrix(Q @ Y.reshape(r, d * D), leg, d, D)
        for l in range(4):
            if l != leg:
                G = _scale_leg(G, l, _inv(lams[legb[site][l]]))
        gammas[site] = G / np.linalg.norm(G)
    return gammas, lams


def su_step(gammas, lams, g, table):
    """one Trotter step (every bond in table order) -> (gammas, lams, delta)"""
    delta = 0.0
    for b in range(len(table)):
        old = lams[b]
        gammas, lams = bond_update(gammas, lams, b, g, table)
        delta = max(delta, float(np.linalg.norm(lams[b] - old)))
    return gammas, lams, delta


def simple_update(gammas, lams, g, max_steps, tol, table):
    """steps until delta < tol or max_steps -> (gammas, lams, steps done, last delta)"""
    steps, delta = 0, float("inf")
    while steps < max_steps:
        gammas, lams, delta = su_step(gammas, lams, g, table)
        steps += 1
        if delta < tol:
            break
    return gammas, lams, steps, delta


def bond_rdm(gammas, lams, b, table):
    """two-site RDM of bond b in the SU environment (lambda on every outer leg of ket and bra), layout [i, i*, j, j*], unit
    trace: the dense pair state psi[p, outer_i, q, outer_j] contracted with its conjugate over the six outer legs."""
    legb = leg_bonds(table)
    i, li, j, lj = table[b]
    Ti = np.moveaxis(_with_outer(gammas[i], i, li, lams, legb), li + 1, -1)      # [p, o, o, o, k]
    Tj = np.moveaxis(_with_outer(gammas[j], j, lj, lams, legb), lj + 1, -1)
    psi = np.einsum("pabck,k,qefgk->pabcqefg", Ti, np.asarray(lams[b]), Tj)
    rho = np.einsum("pabcqefg,PabcQefg->pPqQ", psi, np.conj(psi))
    return rho / np.einsum("iijj->", rho)


def bond_contraction(gammas, lams, b, table):
    """the bond's dense two-site tensor (Gamma_i with outer lambdas) lambda_b (Gamma_j with outer lambdas) as a
    [(p, outer_i), (q, outer_j)] matrix."""
    legb = leg_bonds(table)
    i, li, j, lj = table[b]
    Ti = np.moveaxis(_with_outer(gammas[i], i, li, lams, legb), li + 1, -1)
    Tj = np.moveaxis(_with_outer(gammas[j], j, lj, lams, legb), lj + 1, -1)
    psi = np.einsum("pabck,k,qefgk->pabcqefg", Ti, np.asarray(lams[b]), Tj)
    n = psi.shape[0] * psi.shape[1] ** 3
    return psi.reshape(n, n)


def to_unit_cell_tensors(gammas, lams, table):
    """A, B, C with sqrt(lambda) absorbed on every virtual leg (each bond's lambda split evenly between its two ends)."""
    legb = leg_bonds(table)
    out = []
    for site, G in enumerate(gammas):
        T = G
        for l in range(4):
            T = _scale_leg(T, l, np.sqrt(np.asarray(lams[legb[site][l]], dtype=np.float64)))
        out.append(T)
    return out
