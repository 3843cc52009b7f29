"""How much do the six concurrent side chains slow each other down?  Times one BP iteration (device resident, every side
program one CUDA graph) with 1, 2, 3, 6 sides active.     usage: python tools/side_timing.py D N [--one-plain]
--one-plain: run side D once more with graphs off (what an `ncu` launch list of ONE chain wants: KBP_GRAPHS=0 ncu ... this)."""
import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
from kagomeperiodicbp_b200 import belief_propagation as bp
from kagomeperiodicbp_b200.containers import BPConfig, UnitCell
from kagomeperiodicbp_b200.lattice import BLOCK_SIDES_CCW
from kagomeperiodicbp_b200.runtime import get_engine

D, N = int(sys.argv[1]), int(sys.argv[2])
B = int(sys.argv[3]) if len(sys.argv) > 3 and sys.argv[3].isdigit() else 1        # unit cells batched into every launch
cfg = BPConfig(trunc_dim=2 * D * D, msg_diff_terminate=1e-6, damping=0.1, init_msg="UQ")
cell = UnitCell.random(2, D, seed=0)
msgs = bp.initial_messages(D, N, "UQ")
cache = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpurun_out", f"msgs_D{D}_N{N}.npz")
if os.path.exists(cache):      # steady-state messages of an earlier run: nothing else gets profiled
    from kagomeperiodicbp_b200.containers import Message
    from kagomeperiodicbp_b200.mps import MPS
    z = np.load(cache)
    msgs = {s: Message(MPS.from_sites([z[f"{s}_{k}"] for k in range(2 * N - 1)]), msgs[s].orientation) for s in BLOCK_SIDES_CCW}
else:
    for _ in range(2):
        out, msgs, err, _ = bp.bp_step_batch(N, [cell], [msgs], cfg)[0]
    os.makedirs(os.path.dirname(cache), exist_ok=True)
    np.savez(cache, **{f"{s}_{k}": a for s in BLOCK_SIDES_CCW for k, a in enumerate(msgs[s].mps.A)})
shapes = bp._msg_shapes(msgs)
comps = {s: bp.compile_side_program(N, 2, D, s, 2 * D * D, shapes, 0.1) for s in BLOCK_SIDES_CCW}
engs = {s: get_engine(("side", s), 0) for s in BLOCK_SIDES_CCW}
for s in BLOCK_SIDES_CCW:
    comps[s].load(engs[s], B)
    engs[s].upload(0, comps[s].pack_inputs([bp._side_inputs(cell, msgs, comps[s])] * B))
    engs[s].sync()
if "--one-plain" in sys.argv:
    t0 = time.perf_counter()
    comps["D"].run_resident(engs["D"], (-4,))
    engs["D"].sync()
    print(f"side D, host-driven: {(time.perf_counter() - t0) * 1e3:.1f} ms, {engs['D'].launch_count()} launches so far")
    sys.exit(0)
for s in BLOCK_SIDES_CCW:                      # first sight + capture
    for _ in range(2):
        comps[s].run_resident(engs[s], (-4,))
        engs[s].sync()
if os.environ.get("KBP_KTIME"):
    engs["D"].ktime_report("(reset after warm-up)")
for k in (1, 2, 3, 6):
    sides = BLOCK_SIDES_CCW[:k]
    best = 1e9
    if os.environ.get("KBP_KTIME"):                # the probe tables hold one replay
        engs["D"].ktime_report("(reset)")
    for rep in range(1 if os.environ.get("KBP_KTIME") else 3):
        t0 = time.perf_counter()
        host = []
        if "--threads" in sys.argv:                    # one launching thread per side (graph launches of big programs take host time)
            futs = [bp._pool.submit(comps[s].run_resident, engs[s], (-4,)) for s in sides]
            for f in futs:
                f.result()
            host.append(time.perf_counter() - t0)
        else:
          for s in sides:
            h0 = time.perf_counter()
            comps[s].run_resident(engs[s], (-4,))
            host.append(time.perf_counter() - h0)
        if k == 6:
            print("  host time of the six graph launches (ms):", " ".join(f"{1e3*x:.1f}" for x in host))
        for s in sides:
            engs[s].sync()
        best = min(best, time.perf_counter() - t0)
    print(f"{k} side(s) concurrently, {B} cell(s) per launch: {best*1e3:.1f} ms per iteration")
    if os.environ.get("KBP_KTIME"):
        engs["D"].ktime_report(f"{k} side(s)")
print(engs["D"].svd_counters())
