"""Simple update of a random unit cell (Kagome Heisenberg AFM) on the device, then the block-BP energy of the SU cell and,
optionally, full-update ITE from it (as tools/run_ite.py, modes A, B, C x the six edges per sweep).
usage: python tools/run_su.py D N [ite_sweeps_per_dt [dt ...]]"""
import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from kagomeperiodicbp_b200 import belief_propagation as bp
from kagomeperiodicbp_b200 import edge_env, ite_flow
from kagomeperiodicbp_b200.containers import BPConfig, UnitCell
from kagomeperiodicbp_b200.simple_update import simple_update

D, N = int(sys.argv[1]), int(sys.argv[2])
sweeps = int(sys.argv[3]) if len(sys.argv) > 3 else 0
dts = [float(x) for x in sys.argv[4:]] or [0.1, 0.05, 0.02, 0.01]
chi = 2 * D * D + 10
cfg = BPConfig(trunc_dim=2 * D * D, msg_diff_terminate=1e-6, msg_diff_good_enough=1e-5, damping=0.1, init_msg="UQ", max_iterations=50)
t0 = time.perf_counter()
r = simple_update([UnitCell.random(2, D, seed=0)])[0]
print(f"SU: steps per stage {r.steps}, converged {r.converged}, last deltas {['%.2e' % x for x in r.deltas]}, "
      f"SU-environment energy/site {r.energy_per_site:+.6f}  ({time.perf_counter() - t0:.2f} s)", flush=True)
cell = r.unit_cell
msgs, _ = bp.robust_belief_propagation(bp.KagomeTNRepeatedUnitCell(cell, N), None, cfg)
print(f"block BP (N={N}, chi={chi}) energy/site of the SU cell {ite_flow.measure_energies(cell, msgs, N, chi, mode='A').mean_energy:+.6f}",
      flush=True)
steps = 0
for dt in dts if sweeps else []:
    for sw in range(sweeps):
        for mode in edge_env.MODES:
            order = [(e, dt) for e in edge_env.EDGES]
            cell, msgs, _, _ = ite_flow.ite_per_mode(cell, msgs, N, mode, order, cfg, chi)
            steps += len(order)
        m = ite_flow.measure_energies(cell, msgs, N, chi, mode="A")
        print(f"ITE dt {dt:g} sweep {sw}: energy/site {m.mean_energy:+.6f}  ({steps} edge updates, {time.perf_counter() - t0:.1f} s)",
              flush=True)
