"""How long does the UNMODIFIED reference (oracle/_ref, its own FP32 kernels) take per EventDrivenMap::ComputeF on this
GPU?  edm_ref_time_compute_f of the wrapper loops over the reference's own ComputeF (which ends in a blocking copy).
Measurement helper, not product."""
import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
from oracle import ref_py
import bench
if not ref_py.available():
    sys.exit("oracle/_ref/libedm_ref.so is missing (built where B200_REFERENCE_DIR names the reference)")
z0 = np.array(bench.Z_DRIVER, np.float64)
for N in (1024, 512):
    ms = ref_py.time_compute_f(z0, bench.BETA, 1000, N=N, warm=3, reps=10)
    print(f"reference (unmodified, FP32 kernels), R=1000 N={N}: {ms:.2f} ms per ComputeF", flush=True)
