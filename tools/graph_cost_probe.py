import sys, time, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
from libmultiviewnative_b200 import load
lib = load()
for dims in [(128,128,128),(256,256,256)]:
    rng = np.random.default_rng(0)
    img = (rng.random(dims, dtype=np.float32) + 1)
    w = np.full(dims, 0.5, np.float32); k = rng.random((9,9,9), dtype=np.float32); k /= k.sum()
    with lib.plan(dims, 6, 0) as p:
        for v in range(6): p.set_view(v, img, w, k, k)
        p.set_psi(img); p.iterate(2, 0.006, 1e-4); p.synchronize()
        for n in (3, 3, 3):
            t0 = time.perf_counter(); dev = p.iterate(n, 0.006, 1e-4); wall = (time.perf_counter()-t0)*1e3
            print(dims, 'iterate(%d): device %.3f ms wall %.3f ms' % (n, dev, wall))
