#!/usr/bin/env python
"""Headline benchmark: block-BP message updates per second on the periodic Kagome block, D=4 (BASELINE.json metric), one
process per GPU.

A "step" is ONE BP iteration of one unit cell per chain slot: the six outgoing block messages (six boundary-MPS chains with
per-swallow truncation + normalise + overlap + damping), i.e. 6 message updates per unit cell.  Every side program is ONE
CUDA graph on its own stream (the data-dependent loops of the truncated SVDs are conditional graph nodes), so a step is six
graph launches from one host thread.

  --config C3 (default)  D=4, N=6  (BASELINE.json configs[2]; fits one GPU)        C1: D=2,N=2   C2: D=3,N=3
           C4            D=6, N=2  (chi_bp = 72 stress)                             C5: ensemble, 8 cells per GPU, D=4, N=3
  --gpus N (torchrun)    default sharding "cells": every rank runs the same step on its own, differently seeded unit cells
                         (weak scaling, no data-path collective);  --shard sides: the six sides of ONE cell over the ranks with
                         one NCCL all-gather of the new messages per iteration on device buffers (strong scaling, C3's wording)

  value     message updates/s, inputs resident in HBM
  e2e       same metric through the public API call bp_step_batch(...) with HOST buffers (pack + H2D + run + D2H timed)
  roofline  FP64 tensor (DMMA) roofline: ALL-OPS algorithmic flops of the step (SURVEY 8d conventions: what the reference's
            algorithm costs) / the device-timed step / cuBLAS DGEMM peak measured here; `executed_tflops` is what the kernels
            really execute (the subspace-iteration SVD does ~10x fewer flops than the full SVD the convention counts)
  parity    the device result of the timed workload against the oracle on the same inputs (overlap defect of the side-D
            message when the oracle chain fits the CPU budget) + size-independent properties + a full D=4, N=2 step
  cpu_baseline  the numpy oracle (port of the reference path, exact-SVD branch) on this box's host cores, bounded sample
  ite       second headline metric ("ms per ITE step"): one loop body of ite_per_mode, wall clock on rank 0
`--dump-outputs DIR` writes what the last timed step returned on rank 0 (every unit cell's new messages and errors) as
DIR/<name>.npy, so that two builds can be compared output for output on the same seeded inputs.
`--impl reference` times that CPU port as the reference arm: a step there is a BOUNDED SAMPLE (a prefix of one chain's swallow
order on steady-state messages); value = fraction of a message done / measured seconds, ms_per_step = measured, no extrapolation.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "bp_message_updates_per_s"
UNIT = "msg/s"
CONFIGS = {"C1": dict(D=2, N=2, batch=1), "C2": dict(D=3, N=3, batch=1), "C3": dict(D=4, N=6, batch=1),
           "C4": dict(D=6, N=2, batch=1), "C5": dict(D=4, N=3, batch=8)}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--config", default="C3", choices=sorted(CONFIGS), help="BASELINE.json configuration (sets D, N, batch)")
    ap.add_argument("--D", type=int, default=None)
    ap.add_argument("--N", type=int, default=None)
    ap.add_argument("--batch", type=int, default=None, help="unit cells per GPU batched into every launch")
    ap.add_argument("--damping", type=float, default=0.1)
    ap.add_argument("--shard", default="cells", choices=("cells", "sides"))
    ap.add_argument("--ensemble", type=int, default=8, help="unit cells per launch of the extra ensemble measurement at N=1 (0 = skip)")
    ap.add_argument("--ensemble-N", type=int, default=3)
    ap.add_argument("--ite-steps", type=int, default=3, help="ITE steps timed on rank 0 at N=1 (block size min(N, 3)); 0 = skip")
    ap.add_argument("--seed-offset", type=int, default=0, help="first unit-cell seed of rank 0 (diagnostics: rank r of a multi-GPU run uses seed r * batch)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--cpu-budget-s", type=float, default=25.0)
    ap.add_argument("--parity-budget-s", type=float, default=100.0, help="run the full oracle chain for the parity check if it is estimated to fit")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed (rank 0) as DIR/<name>.npy, float64")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    c = CONFIGS[a.config]
    a.D = c["D"] if a.D is None else a.D
    a.N = c["N"] if a.N is None else a.N
    a.batch = c["batch"] if a.batch is None else a.batch
    return a


L2_NOTE = "512 MiB buffer rewritten between timed iterations (L2 flush)"
SHARDING_CELLS = "independent unit cells per rank, no data-path collective"


def config_dict(a, sharding=SHARDING_CELLS, batch=None):
    """the `config` object of the JSON line -- the same for the GPU arm and for the reference arm of the same invocation"""
    from kagomeperiodicbp_b200 import contraction_order
    return {"workload": workload_name(a), "baseline_config": a.config, "unit_cells_per_gpu": a.batch if batch is None else batch, "sharding": sharding,
            "l2": L2_NOTE, "swallows_per_message": len(contraction_order.kagome_order(a.N, "D", "ToMessage")) - 1}


def workload_name(a):
    n_s = 3 * (3 * a.N * a.N - 3 * a.N + 1)
    return (f"Kagome Heisenberg-PEPS block BP, D={a.D}, block N={a.N} ({n_s} sites, 6 messages x {2 * a.N - 1} MPS sites), "
            f"chi_bp={2 * a.D * a.D}, damping={a.damping}, complex128")


DUMP_LIMIT_BYTES = 60_000_000          # array data of one --dump-outputs directory: under 64 MB with the .npy headers


def step_arrays(results, damping):
    """per unit cell what bp_step_batch returns: the outgoing message of every side, the damped next message (damping only),
    the message error and the truncation error."""
    from kagomeperiodicbp_b200.lattice import BLOCK_SIDES_CCW
    arrays = {}
    for ci, (out_msgs, next_msgs, err, trunc) in enumerate(results):
        kinds = [("out", out_msgs)] + ([("next", next_msgs)] if damping else [])
        for kind, msgs in kinds:
            for s in BLOCK_SIDES_CCW:
                for k, t in enumerate(msgs[s].mps.A):
                    arrays[f"cell{ci}_{kind}_{s}_site{k:02d}"] = t
        arrays[f"cell{ci}_error"] = np.float64(err)
        arrays[f"cell{ci}_trunc_error"] = np.float64(trunc)
    return arrays


def write_outputs(path, arrays):
    """DIR/<name>.npy in float64, complex arrays with a trailing (real, imaginary) axis.  Above DUMP_LIMIT_BYTES every array
    keeps the same fraction of its elements, flattened, at indices drawn from a fixed seed."""
    arrays = {k: np.asarray(v) for k, v in arrays.items()}
    total = sum(a.size * (16 if np.iscomplexobj(a) else 8) for a in arrays.values())
    frac = min(1.0, DUMP_LIMIT_BYTES / total)
    rng = np.random.default_rng(0)
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        if frac < 1.0 and a.ndim:
            a = a.reshape(-1)[np.sort(rng.choice(a.size, max(1, int(a.size * frac)), replace=False))]
        if np.iscomplexobj(a):
            a = np.stack([a.real, a.imag], axis=-1)
        np.save(os.path.join(path, name + ".npy"), a.astype(np.float64))


# ------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    def __init__(self, dev):
        super().__init__(daemon=True)
        self.dev, self.rows, self.stop_flag = dev, [], False

    def run(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.dev}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if r and r[1].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(self.rows)}


# ------------------------------------------------------------------------------------------------
def oracle_chain(N, D, cell, messages, budget_s, full_if_within_s=0.0, side="D"):
    """run the oracle on the ToMessage chain of `side` (or a prefix of its swallow order) of the workload.
    -> dict(seconds, swallows, total, mps or None, seconds_per_message (extrapolated when a prefix was run))"""
    from kagomeperiodicbp_b200 import block_tn, contraction_order
    from kagomeperiodicbp_b200.lattice import SIDE_ANGLE
    from oracle.bubblecon_np import bubblecon as obub
    msgs = {s: m.mps.A for s, m in messages.items()}
    T, E, A, K, P = block_tn.assemble(N, cell.tensors(), msgs)
    T, E, A = block_tn.connect_corner(N, T, E, A, P, side)
    order = list(contraction_order.kagome_order(N, side, "ToMessage"))
    chi = 2 * D * D
    k0 = min(len(order), 8 + 2 * (2 * N - 1))
    t0 = time.perf_counter()
    obub(T, E, A, SIDE_ANGLE[side], order[:k0], D_trunc=chi, ket_tensors=K)
    t_probe = time.perf_counter() - t0
    est_full = t_probe / k0 * len(order) * 1.5
    if est_full < max(budget_s, full_if_within_s):
        k = len(order)
    else:
        k = min(len(order), max(k0, int(budget_s / (1.5 * t_probe / k0))))
    t0 = time.perf_counter()
    mp = obub(T, E, A, SIDE_ANGLE[side], order[:k], D_trunc=chi, ket_tensors=K, separate_exp=True)
    t = time.perf_counter() - t0
    t_full = t if k == len(order) else t + (t - t_probe) / max(1, k - k0) * (len(order) - k)
    return {"seconds": t, "swallows": k, "total": len(order), "mps": mp if k == len(order) else None, "seconds_per_message": t_full}


def cpu_baseline_entry(r):
    full = r["swallows"] == r["total"]
    return {"value": 1.0 / r["seconds_per_message"], "unit": UNIT, "cores": os.cpu_count(), "kind": "port",
            "sample": f"oracle (numpy port of the reference path, exact-SVD branch) on {r['swallows']}/{r['total']} swallows of one ToMessage chain "
                      f"(side D) of the same workload and inputs, {r['seconds']:.1f} s measured" +
                      ("" if full else f", extrapolated to {r['seconds_per_message']:.1f} s per message by the steady-state cost per swallow"),
            "seconds_per_message": r["seconds_per_message"]}


def parity_block(a, cell, msgs_in, step_result, chain):
    """device result of the timed workload vs the oracle + size-independent properties + a full small step."""
    from helpers import overlap_defect, to_oracle_mps
    from kagomeperiodicbp_b200 import belief_propagation as bp
    from kagomeperiodicbp_b200.containers import BPConfig, UnitCell
    from kagomeperiodicbp_b200.lattice import BLOCK_SIDES_CCW, SIDE_OPPOSITE
    from oracle import bp_np, mps_np
    out_msgs = step_result[0]
    worst_norm, worst_canon = 0.0, 0.0
    for s in BLOCK_SIDES_CCW:
        m = to_oracle_mps(out_msgs[s].mps)
        worst_norm = max(worst_norm, abs(abs(mps_np.mps_inner_product(m, m, True)) - 1.0))
        for t in m.A[1:]:
            M = t.reshape(t.shape[0], -1)
            worst_canon = max(worst_canon, float(np.linalg.norm(M @ M.conj().T - np.eye(t.shape[0]))))
    out = {"tolerance": 1e-10, "workload_unit_norm_defect": worst_norm, "workload_right_canonical_defect": worst_canon,
           "workload_finite": bool(all(np.all(np.isfinite(t)) for s in BLOCK_SIDES_CCW for t in out_msgs[s].mps.A))}
    if chain is not None and chain["mps"] is not None:
        dev = to_oracle_mps(out_msgs[SIDE_OPPOSITE["D"]].mps)
        out["workload_side_D_overlap_defect_vs_oracle"] = overlap_defect(chain["mps"], dev)
    else:
        out["workload_side_D_overlap_defect_vs_oracle"] = None
        out["note"] = "the oracle chain of this workload does not fit the parity budget on this host; see the D=4, N=2 step below"
    # one full BP step at D=4, N=2 (second iteration: full-rank spectra), device vs oracle on the same inputs
    D, N = 4, 2
    c2 = UnitCell.random(2, D, seed=5)
    cfg = BPConfig(trunc_dim=2 * D * D, msg_diff_terminate=1e-6, damping=0.1, init_msg="UQ")
    ocfg = bp_np.BPConfigNP(trunc_dim=2 * D * D, msg_diff_terminate=1e-6, damping=0.1)
    m0 = bp.initial_messages(D, N, "UQ")
    _, nxt, _, _ = bp.bp_step_batch(N, [c2], [m0], cfg)[0]
    o2, n2, e2, _ = bp.bp_step_batch(N, [c2], [nxt], cfg)[0]
    om = {s: to_oracle_mps(nxt[s].mps) for s in BLOCK_SIDES_CCW}
    oo, on, oe = bp_np.bp_step(N, c2.tensors(), om, ocfg)
    out["D4_N2_step_max_overlap_defect_vs_oracle"] = max(max(overlap_defect(oo[s], to_oracle_mps(o2[s].mps)),
                                                             overlap_defect(on[s], to_oracle_mps(n2[s].mps))) for s in BLOCK_SIDES_CCW)
    out["D4_N2_step_error_abs_diff"] = abs(e2 - oe)
    vals = [v for k, v in out.items() if k.endswith("vs_oracle") and v is not None]
    out["ok"] = bool(out["workload_finite"] and worst_norm < 1e-10 and worst_canon < 1e-9 and all(v < 1e-10 for v in vals)
                     and out["D4_N2_step_error_abs_diff"] < 1e-8)
    return out


def ite_metric(a, cpu_spm):
    """ms per ITE step: loop bodies of ite_per_mode (BASELINE.json's second metric) on the device, wall clock, after one
    untimed pass over the same edges (program compilation + graph capture), messages warm as in a running ITE."""
    from kagomeperiodicbp_b200 import belief_propagation as bp
    from kagomeperiodicbp_b200 import edge_env, ite_flow
    from kagomeperiodicbp_b200.containers import BPConfig, UnitCell
    D, N = a.D, min(a.N, 3)
    chi = 2 * D * D + 10
    cfg = BPConfig(trunc_dim=2 * D * D, msg_diff_terminate=1e-6, damping=a.damping, init_msg="UQ")
    uc = UnitCell.random(2, D, seed=0)
    tn = bp.KagomeTNRepeatedUnitCell(uc, N)
    msgs, _ = bp.robust_belief_propagation(tn, None, cfg)
    edges = [edge_env.EDGES[k % 6] for k in range(a.ite_steps)]
    for _ in range(2):                                # untimed passes: first sight + capture of every program
        for e in edges:
            uc, msgs, _, _ = ite_flow.ite_edge_update(uc, msgs, N, "A", e, 1e-2, cfg, chi)
    ts, parts, its, energies = [], [0.0, 0.0, 0.0], [], []
    for e in edges:
        t0 = time.perf_counter()
        uc, msgs, energy, st = ite_flow.ite_edge_update(uc, msgs, N, "A", e, 1e-2, cfg, chi)
        ts.append(time.perf_counter() - t0)
        parts = [parts[0] + st.t_bp, parts[1] + st.t_reduce, parts[2] + st.t_update]
        its.append(st.bp_iterations)
        energies.append(energy)
    out = {"metric": "ms_per_ite_step", "value": 1e3 * float(np.mean(ts)), "unit": "ms", "higher_is_better": False, "steps": len(ts),
           "workload": f"D={D}, block N={N}, chi={chi}, delta_t=1e-2, mode A, edges {edges}",
           "bp_iterations_per_step": its,
           "breakdown_ms": {"bp": 1e3 * parts[0] / len(ts), "reduce_to_edge": 1e3 * parts[1] / len(ts), "rdm_gate_als": 1e3 * parts[2] / len(ts)},
           "edge_energies_after": energies, "device_linalg_calls": ite_flow.backend().calls}
    if cpu_spm is not None:
        out["cpu_baseline_estimate_ms"] = 1e3 * (6 * float(np.mean(its)) + 2) * cpu_spm
        out["cpu_baseline_note"] = "(BP iterations x 6 + 2 ToCore) chains at the oracle's measured seconds per chain of this block size; edge algebra not included"
    return out


def steady_state(a, seed):
    """unit cell + messages after two untimed BP iterations from uniform messages (every program shape in its steady state)."""
    from kagomeperiodicbp_b200 import belief_propagation as bp
    from kagomeperiodicbp_b200.containers import BPConfig, UnitCell
    cfg = BPConfig(trunc_dim=2 * a.D * a.D, msg_diff_terminate=1e-6, damping=a.damping, init_msg="UQ")
    return UnitCell.random(2, a.D, seed=seed), cfg


def run_reference_arm(a, rank):
    """the reference's CPU path (oracle port) on the host cores: each step = a bounded prefix of one chain on the steady-state
    messages of the same workload; nothing is multiplied or extrapolated in `value` / `ms_per_step`."""
    if rank != 0:
        return
    try:                      # torchrun exports OMP_NUM_THREADS=1: give the CPU arm every host thread back
        from threadpoolctl import threadpool_limits
        threadpool_limits(limits=os.cpu_count())
    except Exception:
        pass
    from kagomeperiodicbp_b200 import block_tn, contraction_order
    from kagomeperiodicbp_b200.containers import UnitCell
    from kagomeperiodicbp_b200.lattice import BLOCK_SIDES_CCW, SIDE_ANGLE
    from oracle import bp_np
    from oracle.bubblecon_np import bubblecon as obub
    D, N = a.D, a.N
    chi = 2 * D * D
    cell = UnitCell.random(2, D, seed=0)
    # steady-state message SHAPES (bond chi_bp) with random right-canonical content: the cost of a swallow depends on shapes only
    rng = np.random.default_rng(0)
    L, D2 = 2 * N - 1, D * D
    msgs = {}
    for s in BLOCK_SIDES_CCW:
        sites = []
        for k in range(L):
            dl = 1 if k == 0 else min(chi, D2 ** k, D2 ** (L - k))
            dr = 1 if k == L - 1 else min(chi, D2 ** (k + 1), D2 ** (L - k - 1))
            t = rng.normal(size=(dl, D2, dr)) + 1j * rng.normal(size=(dl, D2, dr))
            sites.append(t / np.linalg.norm(t))
        msgs[s] = sites
    side = "D"
    T, E, A, K, P = block_tn.assemble(N, cell.tensors(), msgs)
    T, E, A = block_tn.connect_corner(N, T, E, A, P, side)
    order = list(contraction_order.kagome_order(N, side, "ToMessage"))
    # size the sample so that the whole arm ends within a few minutes: the cost per swallow grows along the chain (the bonds
    # saturate), so the prefix length is found by doubling until one run takes half of the per-step budget
    per_step_budget = max(2.0, 150.0 / max(1, a.steps + a.warmup))
    k = min(len(order), 8 + 2 * L)
    while True:
        t0 = time.perf_counter()
        obub(T, E, A, SIDE_ANGLE[side], order[:k], D_trunc=chi, ket_tensors=K)
        t_probe = time.perf_counter() - t0
        if k >= len(order) or t_probe > per_step_budget / 2:
            break
        k = min(len(order), 2 * k)
    times = []
    for i in range(a.warmup + a.steps):
        t0 = time.perf_counter()
        mp = obub(T, E, A, SIDE_ANGLE[side], order[:k], D_trunc=chi, ket_tensors=K)
        dt = time.perf_counter() - t0
        if i >= a.warmup:
            times.append(dt)
    if a.dump_outputs:
        write_outputs(a.dump_outputs, {f"chain_{side}_site{j:02d}": t for j, t in enumerate(mp.A)})
    sec = float(np.mean(times))
    frac = k / len(order)                 # messages done per step (the early swallows are cheaper than average: favours the CPU)
    v = frac / sec
    sample = (f"oracle (numpy port of the reference path, exact-SVD branch), {os.cpu_count()} host threads: per step the first {k} of {len(order)} "
              f"swallows of one ToMessage chain (side D), steady-state message shapes (bond {chi}); = {frac:.3f} message updates per step")
    line = {"metric": METRIC, "value": v, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": 1e3 * sec, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "c128", "data": "synthetic", "impl": "reference", "units_per_step": frac,
            "config": config_dict(a),                      # the GPU arm's config of the same invocation (the L2 note does not apply to the CPU)
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": os.cpu_count(), "kind": "port", "sample": sample},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
class SideSet:
    """the six side programs of one workload, inputs resident on their engines."""

    def __init__(self, N, dev, cells, msgs_list, damping, key="side"):
        from kagomeperiodicbp_b200 import belief_propagation as bp
        from kagomeperiodicbp_b200.lattice import BLOCK_SIDES_CCW
        from kagomeperiodicbp_b200.runtime import get_engine
        self.bp, self.sides = bp, BLOCK_SIDES_CCW
        D = cells[0].A.shape[1]
        self.B = len(cells)
        shapes = bp._msg_shapes(msgs_list[0])
        chi = 2 * D * D
        self.comps = {s: bp.compile_side_program(N, 2, D, s, chi, shapes, damping if damping else None) for s in self.sides}
        self.engs = {s: get_engine((key, s), dev) for s in self.sides}
        self.h2d = self.d2h = 0
        self.respec = 0
        for s in self.sides:
            batch = [bp._side_inputs(c, m, self.comps[s]) for c, m in zip(cells, msgs_list)]
            self.comps[s].load(self.engs[s], self.B)
            self.engs[s].upload(0, self.comps[s].pack_inputs(batch))
            self.h2d += self.comps[s].in_elems * 16 * self.B
            self.d2h += self.comps[s].out_elems * 16 * self.B + 8 * bp.N_SLOTS * self.B
            self.engs[s].sync()

    def ready(self):
        return all(self.engs[s].graph_ready(self.comps[s].words) for s in self.sides)

    def step(self):
        bp = self.bp
        if self.ready() and max(len(self.comps[s].words) for s in self.sides) > bp.BIG_GRAPH_WORDS:
            futs = [bp._pool.submit(self.comps[s].run_resident, self.engs[s], (bp.E_SVD_NOCONV,)) for s in self.sides]   # big graphs: the launch
            for f in futs:                                         # call itself takes 20-30 ms of host time each (belief_propagation.py)
                f.result()
        elif self.ready():
            for s in self.sides:                                   # six graph launches from this thread
                self.comps[s].run_resident(self.engs[s], (bp.E_SVD_NOCONV,))
        else:                                                      # first sight: host-driven loops, one thread per side
            futs = [bp._pool.submit(self.comps[s].run_resident, self.engs[s], (bp.E_SVD_NOCONV,)) for s in self.sides]
            for f in futs:
                f.result()
        for s in self.sides:
            self.engs[s].sync()
        for s in self.sides:                                       # speculative-graph protocol (include/kbp.h): part of the step
            self.respec += bool(self.comps[s].verify_resident(self.engs[s], (bp.E_SVD_NOCONV,)))

    def collect(self, config):
        """what the last step left on the engines, per unit cell as bp_step_batch returns it"""
        res = {s: self.comps[s].collect(self.engs[s], self.B) for s in self.sides}
        return self.bp.assemble_step(res, self.B, config)

    def spec_counters(self):
        out = {"host_driven_reruns": self.respec}
        for s in self.sides:
            for k, v in self.engs[s].spec_counters().items():
                out[k] = out.get(k, 0) + v
        return out

    def launches(self):
        return sum(self.engs[s].launch_count() for s in self.sides)

    def gemm_flops(self):
        return sum(self.engs[s].gemm_flops() for s in self.sides)

    def graph_counters(self):
        out = {}
        for s in self.sides:
            for k, v in self.engs[s].graph_counters().items():
                out[k] = out.get(k, 0) + v
        return out

    def svd_counters(self):
        out = {}
        for s in self.sides:
            for k, v in self.engs[s].svd_counters().items():
                out[k] = out.get(k, 0) + v
        return out


def timed_steps(ss, steps, flush, barrier, torch):
    ms_total = 0.0
    for _ in range(steps):
        flush.zero_()                      # L2 flush between timed iterations (512 MiB > 126 MB L2)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        ss.step()
        e1.record()
        torch.cuda.synchronize()
        ms_total += e0.elapsed_time(e1)
    return ms_total / steps


def main():
    a = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if a.impl == "reference":
        run_reference_arm(a, rank)
        return

    import torch
    import torch.distributed as dist
    from kagomeperiodicbp_b200 import belief_propagation as bp
    from kagomeperiodicbp_b200.containers import BPConfig, UnitCell
    from kagomeperiodicbp_b200.lattice import BLOCK_SIDES_CCW

    # stdout carries the ONE JSON line and nothing else
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = local
    D, N, B = a.D, a.N, a.batch
    chi = 2 * D * D
    cfg = BPConfig(trunc_dim=chi, msg_diff_terminate=1e-6, damping=a.damping, init_msg="UQ")
    cells = [UnitCell.random(2, D, seed=a.seed_offset + rank * B + i) for i in range(B)]
    uq = bp.initial_messages(D, N, "UQ")
    msgs_list = [uq] * B
    for _ in range(2):                     # two untimed iterations: messages (and every program shape) reach the steady state
        res = bp.bp_step_batch(N, cells, msgs_list, cfg, device=dev)
        msgs_list = [r[1] for r in res]
    ss = SideSet(N, dev, cells, msgs_list, a.damping)
    flush = torch.empty(512 * 1024 * 1024 // 4, dtype=torch.float32, device="cuda")

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # untimed priming (not the warm-up): first sight of the programs is host-driven, the second run captures the graphs
    for _ in range(3):
        if ss.ready() and ss.graph_counters()["graph_replays"] >= 6:
            break
        ss.step()
    for _ in range(a.warmup):
        ss.step()
    sampler = ClockSampler(dev)
    sampler.start()
    barrier()
    l0, g0, f0 = ss.launches(), ss.graph_counters(), ss.gemm_flops()
    ms_step = timed_steps(ss, a.steps, flush, barrier, torch)
    last_step = ss.collect(cfg) if a.dump_outputs and rank == 0 else None
    n_launch = ss.launches() - l0
    executed_flops = (ss.gemm_flops() - f0) / a.steps
    g1 = ss.graph_counters()
    barrier()
    # ---- end to end through the public API with host buffers
    bp.bp_step_batch(N, cells, msgs_list, cfg, device=dev)
    t_e2e = 0.0
    last = None
    for i in range(a.steps):
        flush.zero_()
        barrier()
        t0 = time.perf_counter()
        last = bp.bp_step_batch(N, cells, msgs_list, cfg, device=dev)
        torch.cuda.synchronize()
        t_e2e += time.perf_counter() - t0
    ms_e2e = 1e3 * t_e2e / a.steps
    # ---- sides sharded over the ranks: one all-gather of the new messages per iteration (config C3)
    ms_sharded, gather_bytes = None, 0
    if a.shard == "sides" and world > 1:
        from kagomeperiodicbp_b200 import parallel
        sh = parallel.ShardedSides(N, cells[0], msgs_list[0], cfg, rank, world, dev, engine_key="sharded")
        for _ in range(a.warmup + 2):
            sh.step()
        tot = 0.0
        for i in range(a.steps):
            flush.zero_()
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            err, trunc, _ = sh.step()
            e1.record()
            torch.cuda.synchronize()
            tot += e0.elapsed_time(e1)
        ms_sharded = tot / a.steps
        gather_bytes = sh.gather_bytes
        if a.dump_outputs and rank == 0:
            last_step = [sh.messages() + (err, trunc)]
    if last_step is not None:
        write_outputs(a.dump_outputs, step_arrays(last_step, a.damping))
    sampler.stop_flag = True
    sampler.join(timeout=2)

    ms_ranks = [ms_step]
    if world > 1:
        allms = [torch.zeros(1, device="cuda", dtype=torch.float64) for _ in range(world)]
        dist.all_gather(allms, torch.tensor([ms_step], device="cuda", dtype=torch.float64))
        ms_ranks = [float(x[0]) for x in allms]           # every rank works on its own unit cell (different spectra): the step is their max
        t = torch.tensor([ms_step, ms_e2e, ms_sharded or 0.0], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_step, ms_e2e = float(t[0]), float(t[1])
        ms_sharded = float(t[2]) if ms_sharded is not None else None
        tl = torch.tensor([n_launch], device="cuda", dtype=torch.int64)
        dist.all_reduce(tl)
        n_launch = int(tl[0])
    units = 6 * B * world
    value = units / (ms_step * 1e-3)
    e2e_value = units / (ms_e2e * 1e-3)
    scaling, sharding = "weak", SHARDING_CELLS
    if ms_sharded is not None:
        units, scaling = 6, "strong"
        value = e2e_value = units / (ms_sharded * 1e-3)
        ms_step = ms_e2e = ms_sharded
        sharding = (f"six block sides of one unit cell round-robin over {world} ranks, one NCCL all-gather of {gather_bytes} B per "
                    f"iteration straight between the ranks' device arenas")

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": scaling, "vs_baseline": None, "dtype": "c128",
            "data": "synthetic",
            "config": config_dict(a, sharding, B),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(ss.h2d), "d2h_bytes_per_step": int(ss.d2h), "ms_per_step": ms_e2e},
            "ms_per_step_by_rank": ms_ranks,
            "gpu_launches": int(n_launch),
            "graph_launches": int(g1["graph_replays"] - g0["graph_replays"]) * (world if world > 1 else 1),
            "host_launches_per_step": (g1["graph_replays"] - g0["graph_replays"]) / a.steps,
            "clocks": sampler.summary()}

    if rank == 0:
        total_flops = sum(ss.comps[s].flops for s in BLOCK_SIDES_CCW) * B
        svd_flops = sum(4.0 * (14.0 * max(m, n) * min(m, n) ** 2 + 8.0 * min(m, n) ** 3) for s in BLOCK_SIDES_CCW
                        for (m, n, k) in ss.comps[s].meta["svd_shapes"]) * B
        # measured FP64 peak: cuBLAS DGEMM 4096^3 via torch (library call, used only as the denominator)
        x = torch.randn(4096, 4096, dtype=torch.float64, device="cuda")
        torch.matmul(x, x)
        best = 1e9
        for _ in range(5):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            torch.matmul(x, x)
            e1.record()
            torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1))
        del x
        peak = 2 * 4096 ** 3 / (best * 1e-3) / 1e12
        achieved = total_flops / (ms_step * 1e-3) / 1e12
        traffic, traffic_src = None, None
        tf = os.path.join(ROOT, "profiles", "r02_ncu_traffic.json")
        if os.path.exists(tf):
            tj = json.load(open(tf))
            traffic, traffic_src = tj.get("dominant_kernel_dram_bytes_per_launch"), tj.get("source")
        paths = ss.svd_counters()
        paths.update(ss.spec_counters())
        line["roofline"] = {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                            "traffic": traffic, "traffic_source": traffic_src,
                            "kernel": "whole BP iteration; dominant family = truncated SVD by subspace iteration (zgemm_dmma_kernel + chol_kernel + "
                                      "trsm_kernel per iteration, svd_cluster_kernel Rayleigh-Ritz)",
                            "definition": "ALL-OPS algorithmic flops of the step (shape-only dry run of the reference's swallow program, SURVEY 8d "
                                          "conventions, full-SVD count) / device-timed step / measured FP64 peak: an algorithm-equivalent rate",
                            "peak_source": "cuBLAS DGEMM 4096^3 FP64 measured in this run (MEASURED_PEAKS.json carries no FP64 figure)",
                            "algorithmic_flops_per_step": total_flops, "svd_algorithmic_flops_per_step": svd_flops,
                            "executed_dmma_flops_per_step": executed_flops,
                            "executed_dmma_tflops": executed_flops / (ms_step * 1e-3) / 1e12,
                            "executed_dmma_frac_of_peak": executed_flops / (ms_step * 1e-3) / 1e12 / peak,
                            "executed_note": "real flops the ZGEMM launches of the timed steps executed on the FP64 tensor pipe (6 m n k per complex "
                                             "product, 3M form; this rank; one-SM kernels -- Cholesky, Jacobi, triangular solve -- not included): the "
                                             "subspace iteration does a fraction of the flops of the full SVDs the algorithmic count assumes",
                            "svd_paths": paths}
        if world == 1:
            # per-opcode device time of one host-driven, instrumented repetition (events around every op; six streams overlap)
            for s in BLOCK_SIDES_CCW:
                ss.engs[s].profile_enable(True)
            ss.step()
            ms = np.zeros(16)
            cnt = np.zeros(16, dtype=np.int64)
            for s in BLOCK_SIDES_CCW:
                m_, c_ = ss.engs[s].profile_read()
                ms += m_
                cnt += c_
                ss.engs[s].profile_enable(False)
            line["roofline"]["op_time_ms_host_driven"] = {k: float(ms[i]) for k, i in (("permute", 1), ("gemm", 2), ("qr", 3), ("svd", 4), ("normalize", 5), ("embed", 6), ("zero", 7), ("eye", 10))}
            line["roofline"]["op_counts"] = {k: int(cnt[i]) for k, i in (("permute", 1), ("gemm", 2), ("qr", 3), ("svd", 4))}
        chain = None
        if world == 1 and not a.no_cpu_baseline:
            chain = oracle_chain(N, D, cells[0], msgs_list[0], a.cpu_budget_s, 0.0 if a.no_parity else a.parity_budget_s)
            line["cpu_baseline"] = cpu_baseline_entry(chain)
        if world == 1 and not a.no_parity:
            line["parity"] = parity_block(a, cells[0], msgs_list[0], last[0], chain)
        if world == 1 and a.ensemble > 1 and B == 1 and D <= 4:
            # BASELINE config C5: an ensemble of independent unit cells batched into every launch (same programs, nb chains)
            E, EN = a.ensemble, min(a.ensemble_N, N)
            ecells = [UnitCell.random(2, D, seed=100 + i) for i in range(E)]
            emsgs = [bp.initial_messages(D, EN, "UQ")] * E
            for _ in range(2):
                emsgs = [r[1] for r in bp.bp_step_batch(EN, ecells, emsgs, cfg, device=dev)]
            es = SideSet(EN, dev, ecells, emsgs, a.damping, key="ens")
            for _ in range(4):
                es.step()
            ems = timed_steps(es, 3, flush, barrier, torch)
            one = SideSet(EN, dev, ecells[:1], emsgs[:1], a.damping, key="ens1")   # own engines: nothing learned from the batch
            for _ in range(4):
                one.step()
            oms = timed_steps(one, 3, flush, barrier, torch)
            line["ensemble"] = {"workload": f"D={D}, block N={EN}", "unit_cells_per_gpu": E, "ms_per_step": ems, "value": 6 * E / (ems * 1e-3), "unit": UNIT,
                                "one_cell_ms_per_step": oms, "one_cell_value": 6 / (oms * 1e-3), "throughput_gain_over_one_cell": (6 * E / ems) / (6 / oms),
                                "note": "independent unit cells as extra chains of the same launches; chains leave the subspace loop individually"}
        if world == 1 and a.ite_steps > 0 and D <= 4:
            spm = None
            if "cpu_baseline" in line:
                spm = line["cpu_baseline"]["seconds_per_message"]
                if min(N, 3) != N:
                    c3 = oracle_chain(min(N, 3), D, cells[0], bp.initial_messages(D, min(N, 3), "UQ"), 10.0)
                    spm = c3["seconds_per_message"]
            line["ite"] = ite_metric(a, spm)
        sys.stdout.flush()
        os.write(json_fd, (json.dumps(line) + "\n").encode())
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
