import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench, piml_b200 as P
from scripts.bench_stages import timeit
dev = torch.device("cuda")
N = 100000
p, v, ds, dest, _ = [x.to(dev) for x in bench.synthetic_crowd(N)]
model = P.MLAPM(**bench.MLAPM_KW)
for rows in (12500, 25000, 50000, 100000):
    ms = timeit(lambda: model.advance(p, v, ds, dest, bench.DT, bench.RADIUS, rows=(0, rows)), iters=10)
    print(f"rows={rows}: {ms:.3f} ms  ({rows*N/ms/1e9:.1f} Gpairs/s, ideal share of 9.49 ms: {9.49*rows/N:.3f})")
