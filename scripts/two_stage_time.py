"""One own-path solve for profilers / traces:
python scripts/two_stage_time.py n mode(6 all vectors | 7 smallest half | 8 values only) [one_stage(0 | 1)] [reps]"""
import ctypes as C
import sys

import numpy as np

sys.path.insert(0, ".")
from sclens_b200 import Handle  # noqa: E402
from sclens_b200._lib import ptr  # noqa: E402

n, mode = int(sys.argv[1]), int(sys.argv[2])
one_stage = int(sys.argv[3]) if len(sys.argv) > 3 else 0
reps = int(sys.argv[4]) if len(sys.argv) > 4 else 1
with Handle() as h:
    h._ck(h.lib.scl_debug_force_one_stage(one_stage))
    for _ in range(reps):
        ms = C.c_double()
        h._ck(h.lib.scl_bench_syevd(h.h, n, mode, 1, n // 2 + 65, C.byref(ms)))
        st = np.zeros(8)
        h.lib.scl_debug_last_solve(h.h, ptr(st, C.c_double))
        print(f"n={n} mode={mode} one_stage={one_stage}: {ms.value:.1f} ms; stages {[round(float(x), 1) for x in st]}", flush=True)
