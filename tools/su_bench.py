"""Throughput of the simple-update kernel (KBP_OP_SU): CUDA-event time of one launch of `steps` SU steps (tol = 0, so every
chain runs them all) for D in {2, 4, 6} and nb in {1, 148, 1024} cells, after a warm-up launch; `steps` is sized so that the
timed launch lasts over one second.  The numpy oracle (oracle/su_np.py) on a few cells on the host is the CPU baseline, timed
as measured (no extrapolation).  Writes one JSON file.
usage: python tools/su_bench.py [--out profiles/su_bench.json] [--target-s 1.2]"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np

from kagomeperiodicbp_b200 import ite
from kagomeperiodicbp_b200 import simple_update as su
from kagomeperiodicbp_b200.containers import UnitCell
from kagomeperiodicbp_b200.runtime import get_engine
from oracle import su_np


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = (x.strip() for x in out.split(","))
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:                      # the measurement itself does not depend on it
        return {"error": str(e)}


def time_device(D, nb, target_s):
    cells = [UnitCell.random(2, D, seed=s) for s in range(nb)]
    lam0 = np.full((6, D), 1.0 / np.sqrt(D))
    batch = [{"A": c.A, "B": c.B, "C": c.C, "lam": lam0} for c in cells]
    eng = get_engine(("su-bench", D, nb))
    h = np.ascontiguousarray(ite.heisenberg_afm()).tobytes()

    def timed(steps):
        comp = su._compiled(2, D, ((0.05, steps),), 0.0, h)
        comp.launch(eng, batch)                  # load, upload, warm-up launch
        eng.sync()
        eng.timer_start()
        comp.run_resident(eng)
        ms = eng.timer_stop_ms()
        slots = eng.slots()
        assert np.all(slots[:, 0] == steps) and np.all(slots[:, 2] == 0), slots[:, :3]
        return ms

    steps = 2
    ms = timed(steps)
    steps = max(steps, int(np.ceil(steps * target_s * 1e3 / ms)))
    ms = timed(steps)
    bonds = nb * steps * 6
    return {"D": D, "nb": nb, "steps": steps, "ms": ms, "cell_steps_per_s": nb * steps / (ms * 1e-3),
            "us_per_bond_update": ms * 1e3 / bonds, "us_per_bond_update_per_cell": ms * 1e3 / (steps * 6)}


def time_host(D, cells=2, steps=2):
    g = ite.g_from_exp_h(ite.heisenberg_afm(), 0.05)
    t0 = time.perf_counter()
    for s in range(cells):
        c = UnitCell.random(2, D, seed=s)
        su_np.simple_update(list(c.tensors()), [np.full(D, 1 / np.sqrt(D))] * 6, g, steps, 0.0, su.bond_table())
    dt = time.perf_counter() - t0
    return {"D": D, "cells": cells, "steps": steps, "s": dt, "cell_steps_per_s": cells * steps / dt,
            "us_per_bond_update": dt * 1e6 / (cells * steps * 6)}


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/su_bench.json")
    ap.add_argument("--target-s", type=float, default=1.2)
    args = ap.parse_args()
    out = {"card": card(), "device": [], "host_oracle": []}
    for D in (2, 4, 6):
        for nb in (1, 148, 1024):
            r = time_device(D, nb, args.target_s)
            out["device"].append(r)
            print(json.dumps(r), flush=True)
    for D in (2, 4, 6):
        r = time_host(D)
        out["host_oracle"].append(r)
        print(json.dumps(r), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out["card"]))
