import os, sys; sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import armadillocudalinearinterpolation_b200 as B, bench
for prec in ("f64", "f32"):
    for N in (1024, 512):
        m = B.EventDrivenMap([bench.BETA], 1000, noNeurons=N, precision=prec)
        m.EnableTiming(True)
        for _ in range(3): f = m.ComputeF(bench.Z_DRIVER)
        ms = []
        for _ in range(5):
            m.ComputeF(bench.Z_DRIVER); ms.append(m.LastEvolveMs())
        print(prec, N, f"evolve {np.mean(ms):.3f} ms", f, m.LastCounters(), flush=True)
        m.close()
