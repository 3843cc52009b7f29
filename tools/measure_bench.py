"""Measuring an ensemble of unit cells: the per-cell loop (`ite_flow.measure_energies` once per cell: two ToCore chains with a
batch of one, the Core -> Mode -> Edge reduction on the resident backend, one device program per ToEdge contraction) against
the batched call (`ite_flow.measure_energies_batch`: the two ToCore chains and the compiled measurement program with all the
cells in one launch each, or 8 per launch where 32 arenas of the compiled program would exceed 64 GB), for D = 2, N = 2; D = 3, N = 3; D = 4, N = 3 and 1, 8, 32 cells.

Each cell's messages come from batched block BP (chi_BP = 2 D^2, up to `--bp-iterations` iterations: the measurement's work
depends on the message shapes, which are fixed after the first iterations, not on convergence); chi = 2 D^2 + 10 as in
`ensemble.run_ensemble`.  Every (path, shape, number of cells) is warmed up once, then timed with a host clock around whole
calls (both end by reading their results back, i.e. after a device synchronise), repeated until the window lasts at least
`--window-s` seconds.  The per-chain arena of the compiled program comes from its shape-only compile.  Writes one JSON file
with the card's name and power limit read in the same run.
usage: python tools/measure_bench.py [--out profiles/measure_bench.json] [--window-s 1.0]"""
import argparse
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from su_bench import card

from kagomeperiodicbp_b200 import belief_propagation as bp
from kagomeperiodicbp_b200 import edge_env, ensemble, ite_flow
from kagomeperiodicbp_b200.containers import BPConfig, UnitCell

CONFIGS = ((2, 2), (3, 3), (4, 3))
CELLS = (1, 8, 32)
BATCH_ARENA_GB = 64


def window(fn, min_s):
    """(seconds per call, calls): fn repeated until the window lasts min_s."""
    n, t0 = 0, time.perf_counter()
    while True:
        fn()
        n += 1
        dt = time.perf_counter() - t0
        if dt >= min_s:
            return dt / n, n


def bench_config(D, N, min_s, bp_iterations):
    chi = 2 * D * D + 10
    cells = [UnitCell.random(2, D, seed=1000 + s) for s in range(max(CELLS))]
    cfg = BPConfig(trunc_dim=2 * D * D, msg_diff_terminate=1e-6, damping=0.1, init_msg="UQ", max_iterations=bp_iterations)
    msgs = [r[0] for r in ensemble.belief_propagation_batch(N, cells, cfg, batch=8)]
    shapes = bp._msg_shapes(msgs[0])
    assert all(bp._msg_shapes(m) == shapes for m in msgs)
    tocore = []
    for side in edge_env.CORE_DIRECTIONS["U"][:2]:
        comp = bp.compile_side_program(N, 2, D, side, chi, shapes, None, depth="ToCore", epilogue=False)
        tocore.append([sh for _, _, sh in comp.out_layout])
    mcomp = ite_flow.compile_measurement(N, 2, D, chi, "A", "U", tocore)
    out = {"D": D, "N": N, "chi": chi, "arena_elems_per_chain": mcomp.arena_elems,
           "arena_MB_per_chain": mcomp.arena_elems * 16 / 1e6, "program_ops": mcomp.prog.n_ops, "rows": []}
    for n in CELLS:
        cs, ms = cells[:n], msgs[:n]

        def per_cell():
            return [ite_flow.measure_energies(c, m, N, chi) for c, m in zip(cs, ms)]

        # all the cells in one launch, unless their arenas would exceed BATCH_ARENA_GB: then the default 8 per launch
        batch = n if n * out["arena_MB_per_chain"] <= BATCH_ARENA_GB * 1e3 else 8

        def batched():
            return ite_flow.measure_energies_batch(cs, ms, N, chi, batch=batch)
        ref, got = per_cell(), batched()                       # warm-up of both paths at this shape
        worst = max(abs(a.energies[k] - b.energies[k]) for a, b in zip(ref, got) for k in a.energies)
        t_loop, k_loop = window(per_cell, min_s)
        t_batch, k_batch = window(batched, min_s)
        row = {"cells": n, "cells_per_launch": batch, "per_cell_loop_s": t_loop, "per_cell_loop_calls": k_loop, "batched_s": t_batch, "batched_calls": k_batch,
               "per_cell_loop_cells_per_s": n / t_loop, "batched_cells_per_s": n / t_batch, "speedup": t_loop / t_batch,
               "max_edge_energy_diff": worst}
        out["rows"].append(row)
        print(json.dumps(dict(D=D, N=N, **row)), flush=True)
    return out


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/measure_bench.json")
    ap.add_argument("--window-s", type=float, default=1.0)
    ap.add_argument("--bp-iterations", type=int, default=6)
    args = ap.parse_args()
    res = {"card": card(), "window_s": args.window_s, "bp_iterations": args.bp_iterations, "configs": []}
    print(json.dumps(res["card"]), flush=True)
    for D, N in CONFIGS:
        res["configs"].append(bench_config(D, N, args.window_s, args.bp_iterations))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
