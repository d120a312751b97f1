"""Time the Hades permutation alone: sb200_dbg_hades at 2^22 states, once through a default context (the default
Cauchy MDS qualifies for the small-integer layers) and once through a context whose Cauchy MDS does not (denominators
9..17: the sparse partial rounds), in one process.  Kernel time comes from torch.profiler (CUPTI sees the library's
launches); the call's wall time includes the host<->device copies of the states.

Usage:  python tools/hades_time.py [--n 4194304] [--reps 5]     (needs a GPU)"""
import argparse
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")]
import numpy as np  # noqa: E402
import torch  # noqa: E402
from torch.profiler import ProfilerActivity, profile  # noqa: E402

from schnorr_b200 import Engine, _lib  # noqa: E402
import vectors as V  # noqa: E402

Q = 0x73EDA753299D7D483339D80809A1D80553BDA402FFFE5BFEFFFFFFFF00000001


def run(label, params, states, reps):
    e = Engine([0], params=params)
    try:
        e.dbg_hades(states[:1024])  # module load, first launch
        walls = []
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(reps):
                torch.cuda.synchronize()
                t = time.perf_counter()
                e.dbg_hades(states)
                walls.append(time.perf_counter() - t)
        ks = [ev for ev in prof.events() if ev.device_type == torch.autograd.DeviceType.CUDA and "k_run" in ev.name]
        kms = sorted(ev.device_time / 1e3 for ev in ks)
        n = len(states)
        med = kms[len(kms) // 2]
        print(f"{label:34s} n={n} kernel median {med:8.3f} ms  (min {kms[0]:.3f}, max {kms[-1]:.3f}, {len(kms)} launches)  "
              f"{n / med / 1e3:8.2f} M perm/s   call wall median {sorted(walls)[len(walls) // 2] * 1e3:8.1f} ms", flush=True)
        return med
    finally:
        e.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1 << 22)
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    rs = np.random.RandomState(7)
    states = rs.randint(0, 1 << 32, size=(a.n, 40), dtype=np.uint64).astype(np.uint32)
    states[:, 7::8] &= 0x3FFFFFFF  # < 2^254 < q: canonical words
    p_int = _lib.default_params(_lib.ARK_CUMSUM)
    p_sparse = _lib.default_params(_lib.ARK_CUMSUM)
    p_sparse.view("mds")[...] = np.stack([V.mont(pow(i + j + 9, -1, Q)) for i in range(5) for j in range(5)])
    name = torch.cuda.get_device_name(0)
    print(f"device: {name}", flush=True)
    t_int = run("small-integer layers (default MDS)", p_int, states, a.reps)
    t_sp = run("sparse rounds (1/(i+j+9) MDS)", p_sparse, states, a.reps)
    print(f"kernel time ratio sparse / small-integer: {t_sp / t_int:.3f}", flush=True)


if __name__ == "__main__":
    main()
