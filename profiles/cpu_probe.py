import sys, time, os
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, 'multimodal-fusion-based-pre-routing-timing-prediction-_b200'))
import bench, torch
print('cores', os.cpu_count())
for scale in (10, 4, 2, 1):
    total, gnn_only, n = bench.cpu_step(scale, threads=os.cpu_count())
    t0=time.time(); tt = total(); tg = gnn_only()
    print('scale', scale, 'pins', n, 'total %.2f gnn %.2f'%(tt, tg), flush=True)
