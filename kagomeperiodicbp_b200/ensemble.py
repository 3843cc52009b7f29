"""Ensembles of independent unit cells (random restarts, field sweeps): the replacement of the reference's HTCondor fan-out
(scripts/condor/main_sender.py:60-135 submits one job per (seed, D, N, chi, ...); scripts/condor/worker.py:38-165 runs it
and appends one CSV row with the keys scripts/condor/main_sender.py DEFAULT_RESULT_KEYS_DICT names).

Here the seeds are sharded over the ranks of the process group (no data-path collective: the problems are independent), each
rank batches its cells into the SAME launches (``nb`` chains per kernel, chains leave the data-dependent loops individually),
and rank 0 writes the same CSV columns after one gather of scalars.
"""
from __future__ import annotations

import copy
import csv
import os
import time

import numpy as np

from . import belief_propagation as bp
from . import ite_flow
from .containers import BPConfig, UnitCell

RESULT_KEYS = ["seed", "D", "N", "chi", "energy", "parallel", "path", "method", "exec_time", "bp_iterations", "bp_error"]


def seeds_of_rank(seeds, rank: int, world: int):
    return [s for k, s in enumerate(seeds) if k % world == rank]


def belief_propagation_batch(N: int, cells: list, config: BPConfig, messages_list: list | None = None, device: int = 0, batch: int = 8):
    """block BP to convergence for a list of independent unit cells, ``batch`` cells per launch.  Cells that converged (or were
    deemed failing, src/algo/belief_propagation.py:262-273) drop out of the following iterations.
    -> [(messages, iterations, final_error, success)] in input order."""
    n = len(cells)
    D = cells[0].A.shape[1]
    msgs = [bp.initial_messages(D, N, "UQ" if config.init_msg in ("UQ", "UNIFORM_QUANTUM") else "RQ") if (messages_list is None or messages_list[i] is None)
            else messages_list[i] for i in range(n)]
    errors = [[] for _ in range(n)]
    best = [(np.inf, None)] * n
    out = [None] * n
    active = list(range(n))
    it = 0
    k_fail = config.times_to_deem_failure_when_diff_increases
    while active and (config.max_iterations is None or it < config.max_iterations):
        it += 1
        # group by message shapes (bonds grow during the first iterations; cells of one ensemble stay in step)
        groups: dict = {}
        for i in active:
            groups.setdefault(bp._msg_shapes(msgs[i]), []).append(i)
        still = []
        for shape_key, idx in groups.items():
            for c0 in range(0, len(idx), batch):
                chunk = idx[c0:c0 + batch]
                res = bp.bp_step_batch(N, [cells[i] for i in chunk], [msgs[i] for i in chunk], config, device=device)
                for i, (o, nxt, err, _) in zip(chunk, res):
                    errors[i].append(err)
                    if err < config.msg_diff_terminate:
                        out[i] = (o, it, err, True)
                        continue
                    if err < best[i][0]:
                        best[i] = (err, copy.deepcopy(o))
                    e = errors[i]
                    if len(e) > k_fail and all(a <= b for a, b in zip(e[-k_fail:], e[-k_fail:][1:])):
                        out[i] = (best[i][1], it, best[i][0], False)
                        continue
                    msgs[i] = nxt
                    still.append(i)
        active = still
    for i in active:                                   # iteration budget spent
        out[i] = (best[i][1], it, best[i][0], False)
    if config.hermitize_msgs_when_finished:
        out = [(bp._hermitize_messages(o[0]),) + o[1:] for o in out]
    return out


def run_ensemble(seeds, D: int, N: int, chi_factor: float = 1.0, rank: int = 0, world: int = 1, device: int = 0, batch: int = 8,
                 ite_steps: int = 0, delta_t: float = 1e-2, save_folder: str | None = None, method: int = 3, init: str = "random"):
    """one row per seed: random unit cell (method 3 of scripts/condor/send_ite.py:66-70) -> batched block BP -> `ite_steps` ITE
    edge updates per cell -> energy per site.  ``init="su"``: the rank's random cells first go through one batched simple
    update (simple_update.simple_update, default schedule) and BP starts from the SU cells.  Returns this rank's rows."""
    if init not in ("random", "su"):
        raise ValueError(f"init must be 'random' or 'su', got {init!r}")
    mine = seeds_of_rank(list(seeds), rank, world)
    chi_bp = int(2 * D * D * chi_factor)
    chi = int((2 * D * D + 10) * chi_factor)
    cfg = BPConfig(trunc_dim=chi_bp, msg_diff_terminate=1e-6, msg_diff_good_enough=1e-5, damping=0.1, max_iterations=50, init_msg="UQ")
    t0 = time.perf_counter()
    cells = [UnitCell.random(2, D, seed=s) for s in mine]
    if init == "su" and cells:
        from .simple_update import simple_update
        cells = [r.unit_cell for r in simple_update(cells, device=device)]
    res = belief_propagation_batch(N, cells, cfg, device=device, batch=batch)
    rows = []
    for s, cell, (msgs, its, err, ok) in zip(mine, cells, res):
        t1 = time.perf_counter()
        path = None
        for k in range(ite_steps):
            from .edge_env import EDGES
            cell, msgs, _, st = ite_flow.ite_edge_update(cell, msgs, N, "A", EDGES[k % 6], delta_t, cfg, chi, save=save_folder or False)
            path = st.saved_to or path
        m = ite_flow.measure_energies(cell, msgs, N, chi)
        rows.append({"seed": s, "D": D, "N": N, "chi": chi_factor, "energy": m.mean_energy, "parallel": world > 1, "path": path, "method": method,
                     "exec_time": (time.perf_counter() - t1) + (t1 - t0) / max(1, len(mine)), "bp_iterations": its, "bp_error": err})
    return rows


def gather_rows(rows, world: int, group=None):
    """every rank's rows on rank 0 (a gather of small Python objects: the only communication of an ensemble run)."""
    if world == 1:
        return rows
    import torch.distributed as dist
    buf = [None] * world
    dist.all_gather_object(buf, rows, group=group)
    return [r for part in buf for r in part]


def write_csv(rows, path: str, keys=RESULT_KEYS):
    """header row written as data, then one row per result: what main_sender / worker produce (main_sender.py:129-132)."""
    new = not os.path.exists(path)
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    with open(path, "a", newline="") as f:
        w = csv.DictWriter(f, fieldnames=keys)
        if new:
            w.writerow({k: k for k in keys})
        for r in sorted(rows, key=lambda r: r["seed"]):
            w.writerow({k: r.get(k) for k in keys})
    return path
