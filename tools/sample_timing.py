"""Timing of inverse-CDF sampling at N=30 (qipb200_state_sample) against single-draw soft_measure calls.

The state is an H layer on |0...0> (flat distribution: every chunk is hit, the worst case for the per-draw gathers),
in f64 (16 GiB) and f32 (8 GiB).  Each time is a host clock around the call, which ends in a stream synchronise
(the outcomes are copied back to the host), after one warm-up call; the median of 5 is reported.

    python tools/sample_timing.py [--out profiles/r3_sample_n30.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from rustqip_b200 import circuits  # noqa: E402
from rustqip_b200.state import Context, State  # noqa: E402

KS = [1, 1 << 10, 1 << 16, 1 << 20, 1 << 22]
REPS = 5


def median_ms(fn):
    fn()
    ts = []
    for _ in range(REPS):
        t0 = time.perf_counter()
        fn()
        ts.append((time.perf_counter() - t0) * 1e3)
    return statistics.median(ts)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_sample_n30.json"))
    ap.add_argument("--n", type=int, default=30)
    a = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    n = a.n
    qubits = list(range(n))
    rng = np.random.default_rng(1)
    result = {"n": n, "gpu": gpu[0] if gpu else "unknown", "state": "H layer (flat)", "reps": REPS,
              "timing": "host clock around call + synchronise, median after one warm-up", "rows": []}
    with Context(0) as ctx:
        for dtype in (np.complex128, np.complex64):
            with State(n, dtype, ctx) as st:
                st.set_basis(0)
                st.apply_schedule(circuits.h_layer(n))
                st.sync()
                one = float(rng.random())
                row = {"dtype": np.dtype(dtype).name, "soft_measure_ms": median_ms(lambda: st.soft_measure(qubits, one))}
                for K in KS:
                    draws = rng.random(K)
                    row["sample_ms_K%d" % K] = median_ms(lambda: st.sample(qubits, draws))
                row["sample_K2^20_over_soft_measure"] = row["sample_ms_K%d" % (1 << 20)] / row["soft_measure_ms"]
                result["rows"].append(row)
                print(json.dumps(row), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps({"gpu": result["gpu"], "out": a.out}))


if __name__ == "__main__":
    main()
