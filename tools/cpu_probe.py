import sys, os, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, 'oracle')); sys.path.insert(0, ROOT)
if os.environ.get('WITH_TORCH'): import torch
import dcreg_oracle_c as oc
from dcreg_b200.scenes import make_cylinder, g2_initial_pose
pts = make_cylinder(100_000, seed=42)
sc = oc.Scene(pts, pts)
print('max threads', oc.max_threads(), 'cpu_count', os.cpu_count(), 'affinity', len(os.sched_getaffinity(0)))
for mode in (1, 0):
    for it in (2, 10, 10, 30):
        prm = oc.make_params(max_iterations=it, fixed_iterations=True, kappa_target=10.0, use_weight_derivative=False, thread_mode=mode)
        t0 = time.perf_counter(); sc.icp_run(prm, g2_initial_pose(), want_log=False); dt = time.perf_counter() - t0
        print('mode', mode, 'iters', it, '%.1f ms/iter' % (dt / it * 1e3))
