"""From the block with converged messages to the environment of one edge: the reduction chain

    reduce_full_kagome_to_core   src/algo/tn_reduction/kagome_to_core.py:322-364   (two ToCore boundary contractions, zip of
                                 the overlaps :192-215, the 12 environment tensors in canonical order :235-257, attached to
                                 the 9 core kets :260-318)
    reduce_core_to_mode          src/algo/tn_reduction/core_to_mode.py:16-58
    reduce_mode_to_edge          src/algo/tn_reduction/mode_to_edge.py:250-295  (QR split of the common neighbour :268-275,
                                 or a truncated ToEdge boundary contraction when the mode's centre is not on the edge :166-218)
    EdgeTN canonical order       src/tensor_networks/tensor_network.py:790, 1373  (T_i, T_j = [p, shared, 3 others ccw];
                                 ring = [prev, to-core, next] starting at T_i's first free leg)

What is computed is what the reference computes -- the same two truncated ToCore chains, the same exact contractions, the
same truncated ToEdge chain in the six (mode, edge) cases that have one -- but not how: the reference drives a generic
graph container (ArbitraryTN.contract with random set pops, tensor_network.py:1278-1438); here the 21-node core network is a
fixed topology, read from ``core_tables.json`` (node members, leg names, leg angles, swallow orders: data dumped from the
reference by tools/make_golden_ite.py, independent of D, N and of the tensors), and every tensor contraction / QR goes to
the backend ``B`` (device programs in the product).  Ring bonds are gauge freedom: QR splits and the order in which exact
contractions are done differ from the reference, the resulting RDMs / N_red / updated tensors do not.
"""
from __future__ import annotations

import json
import os
from functools import lru_cache

import numpy as np

from .lattice import get_block

_HERE = os.path.dirname(os.path.abspath(__file__))
MODES = ("A", "B", "C")
EDGES = ("AB", "AC", "BA", "BC", "CA", "CB")          # UpdateEdge.all_options() order (src/containers/imaginary_time_evolution.py)


@lru_cache(maxsize=1)
def tables():
    with open(os.path.join(_HERE, "core_tables.json")) as f:
        return json.load(f)


# ------------------------------------------------------------------------------------------------
# named-leg tensors
# ------------------------------------------------------------------------------------------------
class Node:
    __slots__ = ("t", "legs")

    def __init__(self, t, legs):
        assert t.ndim == len(legs), (t.shape, legs)
        self.t, self.legs = t, list(legs)


def fuse_ket(B, T):
    """double layer of a ket tensor [p, k1..kn] -> [k1 k1*, .., kn kn*] (ket index major, as src/libs/bubblecon.py:303-337)."""
    n = T.ndim
    T2 = B.tensordot(T, T, ([0], [0]), conj_b=True)
    perm = [x for i in range(n - 1) for x in (i, i + n - 1)]
    return B.reshape(B.transpose(T2, perm), [T.shape[i] ** 2 for i in range(1, n)])


def contract(B, a: Node, b: Node) -> Node:
    common = [e for e in a.legs if e in b.legs]
    assert common, (a.legs, b.legs)
    ia, ib = [a.legs.index(e) for e in common], [b.legs.index(e) for e in common]
    t = B.tensordot(a.t, b.t, (ia, ib))
    return Node(t, [e for e in a.legs if e not in common] + [e for e in b.legs if e not in common])


def arrange(B, n: Node, legs) -> Node:
    """transpose / fuse to the requested legs; 'x+y' fuses legs x and y (x major)."""
    atoms, sizes = [], []
    for name in legs:
        parts = name.split("+") if name not in n.legs else [name]
        atoms += parts
        sizes.append(int(np.prod([n.t.shape[n.legs.index(p)] for p in parts])))
    assert sorted(atoms) == sorted(n.legs), (legs, n.legs)
    t = B.transpose(n.t, [n.legs.index(p) for p in atoms])
    return Node(B.reshape(t, sizes), list(legs))


# ------------------------------------------------------------------------------------------------
# block -> core
# ------------------------------------------------------------------------------------------------
def core_site_indices(N: int):
    """block indices of the 9 core sites in the reference's canonical order (sorted, items 2 and 3 swapped:
    kagome_to_core.py:351)."""
    idx = sorted(get_block(N).core_indices())
    assert len(idx) == 9
    idx[2], idx[3] = idx[3], idx[2]
    return idx


CORE_DIRECTIONS = {"U": ("U", "D", 0), "DL": ("DL", "UR", 4), "DR": ("DR", "UL", 8)}   # bottom-up side, top-down side, ring rotation


def core_env_tensors(B, N: int, mps_bottom_up, mps_top_down, direction: str = "U"):
    """zip the two ToCore boundary MPSs (bottom-up ``direction`` / its opposite) outside the core and return the 12 ring
    tensors m0..m11 (kagome_to_core.py:192-257; the ring is rotated by 0 / 4 / 8 places for U / DL / DR, :245-255).
    Inputs: lists of site tensors [Dl, D^2, Dr] of the backend ``B`` (host arrays, or traced tensors of a compiled program).
    The open end bonds are dropped with ``B.reshape``, so no site is read on the host."""
    s = 2 * N - 3
    bu, td = list(mps_bottom_up), list(mps_top_down)
    assert len(bu) == 5 + 2 * s and len(td) == 7 + 2 * s, (len(bu), len(td))
    Lt = None
    for j in range(s):
        a, b = B.transpose(td[-j - 1], (2, 1, 0)), bu[j]
        if Lt is None:
            Lt = B.tensordot(B.reshape(a, a.shape[1:]), B.reshape(b, b.shape[1:]), ([0], [0]))
        else:
            Lt = B.tensordot(B.tensordot(Lt, a, ([0], [0])), b, ([0, 1], [0, 1]))
    bu[s] = B.tensordot(Lt, bu[s], ([1], [0]))
    Rt = None
    for j in range(s):
        a, b = B.transpose(td[j], (2, 1, 0)), bu[-1 - j]
        if Rt is None:
            Rt = B.tensordot(B.reshape(a, a.shape[:2]), B.reshape(b, b.shape[:2]), ([1], [1]))
        else:
            Rt = B.tensordot(B.tensordot(a, Rt, ([2], [0])), b, ([1, 2], [1, 2]))
    td[s] = B.tensordot(Rt, td[s], ([0], [0]))
    ring = bu[s + 2:s + 5] + td[s:s + 7] + bu[s:s + 2]
    k = CORE_DIRECTIONS[direction][2]
    return ring[-k:] + ring[:-k] if k else ring


def core_network(B, N: int, cell, env12):
    """the 21 nodes of the CoreTN keyed by the table's node index: kets as (raw tensor, leg names), ring tensors as Nodes."""
    tb = tables()["core"]
    flavor = {"A": 0, "B": 1, "C": 2}
    kets = {}
    core_idx = core_site_indices(N)
    for k in range(9):
        # repeated unit cell: by flavor; non-repeated block (one tensor per lattice site): the core site's own tensor
        t = cell[flavor[tb[k]["name"]]] if len(cell) == 3 else cell[core_idx[k]]
        kets[k] = (t, list(tb[k]["edges"]))
    envs = {}
    for i in range(12):
        envs[i] = Node(env12[i], list(tb[9 + i]["edges"]))
    return kets, envs


class Core:
    """lazily fused double-layer kets + ring tensors, with name resolution of the reference's composite node names."""

    def __init__(self, B, N, cell, env12):
        self.B = B
        self.kets, self.envs = core_network(B, N, cell, env12)
        self._fused = {}
        tb = tables()["core"]
        self.flavor = {k: tb[k]["name"] for k in range(9)}

    def fused(self, k) -> Node:
        if k not in self._fused:
            T, legs = self.kets[k]
            self._fused[k] = Node(fuse_ket(self.B, T), legs)
        return self._fused[k]

    def node(self, key) -> Node:
        return self.envs[key[1]] if key[0] == "m" else self.fused(key[1])

    def legs_of(self, key):
        return self.envs[key[1]].legs if key[0] == "m" else self.kets[key[1]][1]

    def resolve(self, name: str, exclude: set):
        """member keys of a composite node name such as 'm0+m11+A+m10+m9+C+B' (tokens are in contraction order, so each
        ket letter is the not-yet-used core ket of that flavour adjacent to the members collected so far)."""
        members = []
        for tok in name.split("+"):
            if tok[0] == "m" and tok[1:].isdigit():
                members.append(("m", int(tok[1:])))
                continue
            have = set()
            for key in members:
                have.update(self.legs_of(key))
            cands = [k for k in range(9) if self.flavor[k] == tok and ("k", k) not in exclude and ("k", k) not in members
                     and (not members or have & set(self.kets[k][1]))]
            assert len(cands) == 1, (name, tok, cands)
            members.append(("k", cands[0]))
        return members

    def composite(self, members) -> Node:
        """contract the member nodes exactly.  Greedy pairwise order: always the connected pair whose product is
        smallest (the order is free -- exact contraction -- and a bad one creates intermediates with many open D^2 legs)."""
        nodes = [self.node(k) for k in members]
        while len(nodes) > 1:
            best = None
            for x in range(len(nodes)):
                for y in range(x + 1, len(nodes)):
                    a, b = nodes[x], nodes[y]
                    common = [e for e in a.legs if e in b.legs]
                    if not common:
                        continue
                    size = 1
                    for e, dsz in zip(a.legs, a.t.shape):
                        if e not in common:
                            size *= dsz
                    for e, dsz in zip(b.legs, b.t.shape):
                        if e not in common:
                            size *= dsz
                    if best is None or size < best[0]:
                        best = (size, x, y)
            if best is None:
                raise AssertionError(("disconnected composite", members))
            _, x, y = best
            c = contract(self.B, nodes[x], nodes[y])
            nodes = [n for k, n in enumerate(nodes) if k not in (x, y)] + [c]
        return nodes[0]


# ------------------------------------------------------------------------------------------------
# core -> mode -> edge
# ------------------------------------------------------------------------------------------------
def _site_key(core: Core, tnode, taken):
    """core ket of an EdgeTN site node (flavour letter + its leg names identify it)."""
    for k in range(9):
        if core.flavor[k] == tnode["name"] and sorted(core.kets[k][1]) == sorted(tnode["edges"]) and k not in taken:
            return k
    raise AssertionError(tnode)


def edge_environment(B, N: int, cell, env12, mode: str, edge: str, chi: int, bubblecon_fn=None):
    """-> (Ti, Tj, mps_env[6], info) in the EdgeTN's canonical order; info = {i, j: core kets, perm_i, perm_j}.

    ``bubblecon_fn(T_list, edges_list, angles_list, bubble_angle, swallow_order, D_trunc, ket_tensors) -> list of MPS site
    arrays`` runs the truncated ToEdge contraction (device bubblecon in the product, the numpy oracle in tests)."""
    tb = tables()["modes"][mode]
    et = tb["edges"][edge]
    core = Core(B, N, cell, env12)
    ki = _site_key(core, et["nodes"][0], set())
    kj = _site_key(core, et["nodes"][1], {ki})
    ring_tbl = et["nodes"][2:]
    exclude = {("k", ki), ("k", kj)}
    ring: list = [None] * 6

    if et["bubblecon"] is not None:
        bc = et["bubblecon"]
        # the 13 ModeTN nodes in the reference's order: kets raw, everything else fused [a, D^2, b]
        T_list, used = [], set()
        for n in tb["nodes"]:
            if n["ket"]:
                k = next(k for k in range(9) if core.flavor[k] == n["name"] and core.kets[k][1] == n["edges"])
                T_list.append(core.kets[k][0])
            else:
                T_list.append(arrange(B, core.composite(core.resolve(n["name"], set())), n["edges"]).t)
        sites = bubblecon_fn(T_list, bc["edges"], bc["angles"], bc["bubble_angle"], bc["order"], chi, bc["kets"])
        assert len(sites) == 4
        e01 = B.tensordot(B.reshape(sites[0], sites[0].shape[1:]), sites[1], ([1], [0]))     # [open0, open1, bond]
        e32 = B.tensordot(sites[2], B.reshape(sites[3], sites[3].shape[:2]), ([2], [0]))     # [bond, open2, open3]
        for pos, n in enumerate(ring_tbl):
            if n["name"] == "e-0+e-1":
                ring[pos] = Node(e01, n["edges"])
            elif n["name"] == "e-3+e-2":
                ring[pos] = Node(e32, n["edges"])
            else:
                ring[pos] = arrange(B, core.composite(core.resolve(n["name"], exclude)), n["edges"])
    else:
        members_used = set(exclude)
        qr_pos = {}
        for pos, n in enumerate(ring_tbl):
            if n["name"] in ("Q", "R"):
                qr_pos[n["name"]] = pos
                continue
            mem = core.resolve(n["name"], exclude)
            members_used.update(mem)
            ring[pos] = arrange(B, core.composite(mem), n["edges"])
        # the common neighbour with everything that is left, split in two by QR (any split is a gauge of the ring bond)
        rest = [("k", k) for k in range(9) if ("k", k) not in members_used] + [("m", i) for i in range(12) if ("m", i) not in members_used]
        big = core.composite(rest)
        ql, rl = ring_tbl[qr_pos["Q"]]["edges"], ring_tbl[qr_pos["R"]]["edges"]
        q_out = [e for e in ql if e != "qr_edge"]
        r_out = [e for e in rl if e != "qr_edge"]
        m = arrange(B, big, ["+".join(q_out), "+".join(r_out)]) if len(q_out) > 1 else arrange(B, big, [q_out[0], "+".join(r_out)])
        Qm, Rm = B.qr(m.t)
        q_dims = [big.t.shape[big.legs.index(p)] for name in q_out for p in (name.split("+") if name not in big.legs else [name])]
        r_dims = [big.t.shape[big.legs.index(p)] for name in r_out for p in (name.split("+") if name not in big.legs else [name])]
        q_atoms = [p for name in q_out for p in (name.split("+") if name not in big.legs else [name])]
        r_atoms = [p for name in r_out for p in (name.split("+") if name not in big.legs else [name])]
        qn = Node(B.reshape(Qm, q_dims + [Qm.shape[1]]), q_atoms + ["qr_edge"])
        rn = Node(B.reshape(Rm, [Rm.shape[0]] + r_dims), ["qr_edge"] + r_atoms)
        ring[qr_pos["Q"]] = arrange(B, qn, ql)
        ring[qr_pos["R"]] = arrange(B, rn, rl)

    # canonical leg order of the two sites, ring tensors with the D^2 leg opened to (ket, bra)
    pi, pj = et["perms"][et["nodes"][0]["name"]], et["perms"][et["nodes"][1]["name"]]
    Ti = B.transpose(core.kets[ki][0], [0] + [1 + p for p in pi])
    Tj = B.transpose(core.kets[kj][0], [0] + [1 + p for p in pj])
    D = Ti.shape[1]
    env = []
    for n in ring:
        a, d2, b = n.t.shape
        assert d2 == D * D
        env.append(B.reshape(n.t, (a, D, D, b)))
    # consistency of the ring with the sites' canonical legs
    ti_legs = [core.kets[ki][1][p] for p in pi]
    tj_legs = [core.kets[kj][1][p] for p in pj]
    assert ti_legs[0] == tj_legs[0]
    assert [n.legs[1] for n in ring] == ti_legs[1:] + tj_legs[1:], ([n.legs for n in ring], ti_legs, tj_legs)
    for a, b in zip(ring, ring[1:] + ring[:1]):
        assert a.legs[2] == b.legs[0] and a.t.shape[2] == b.t.shape[0], (a.legs, b.legs)
    return _contiguous(Ti), _contiguous(Tj), env, dict(i=ki, j=kj, perm_i=pi, perm_j=pj, flavors=(core.flavor[ki], core.flavor[kj]))


def _contiguous(t):
    """host arrays are returned C-contiguous; a traced tensor of a compiled program already is."""
    return np.ascontiguousarray(t) if isinstance(t, np.ndarray) else t


def write_back(cell, info, Ti_new, Tj_new):
    """put the updated tensors back into the unit cell in their native leg order
    (src/algo/imaginary_time_evolution/_tn_update.py:141-163)."""
    flavor = {"A": 0, "B": 1, "C": 2}
    cell = list(cell)
    for f, perm, t in ((info["flavors"][0], info["perm_i"], Ti_new), (info["flavors"][1], info["perm_j"], Tj_new)):
        inv = np.argsort(perm)
        cell[flavor[f]] = np.ascontiguousarray(np.transpose(np.asarray(t), [0] + [1 + int(p) for p in inv]))
    return cell
