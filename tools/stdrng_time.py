"""What drawing the nonces costs: the host recipe (numpy ChaCha12 blocks, sb200_scalars_from_wide, then sb200_sign) against
the device-side draw (sb200_sign_stdrng), in one process on one GPU, the two paths alternated over several repetitions.

  (a) sb200_stdrng_random alone, 2^22 JubJubScalar draws, device-resident output: the generation kernel's time
      (CUDA events around back-to-back calls).
  (b) sign 2^20 and 2^22 from pinned host buffers.  Path 1 (host draw) is bench.py's c3 recipe: bench.stdrng_nonces
      (numpy ChaCha12 in 2^20-block steps, reduced on the device by sb200_scalars_from_wide from pageable memory), the
      nonces copied into the pinned nonce buffer, then sb200_sign.  Path 2 is sb200_sign_stdrng on the same sk / msg
      buffers.  Path 1's three parts are timed separately.  u, R and c must be byte-identical.
  (c) the same for sign_double at 2^20.
  (d) bench.py's e2e_typed leg (build/bench_typed: the typed C++ API, whose batch signers now draw on the device) at
      2^20 and 2^22 on this build, printed next to the committed profiles/bench_typed_r02b.json of an earlier build:
      a comparison across builds, not an A/B in one process.

Prints one JSON object (also written to --out) with the card's name and power limit.
Usage:  python tools/stdrng_time.py [--reps 5] [--out FILE]     (needs a GPU)"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")]
sys.dont_write_bytecode = True
import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402  (the c3 nonce recipe: seed_from_u64, stdrng_nonces)
from schnorr_b200 import Engine  # noqa: E402
from schnorr_b200._lib import DEVICE_PTRS, StdRngPos  # noqa: E402

SEED = 0xC3


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip() or q.stderr.strip()}


def pinned(shape):
    t = torch.empty(shape, dtype=torch.int32, pin_memory=True)
    return t, t.numpy().view(np.uint32)


def stats(xs):
    s = sorted(xs)
    return {"median_ms": round(s[len(s) // 2], 3), "min_ms": round(s[0], 3), "max_ms": round(s[-1], 3), "reps": len(s)}


def time_generation(eng, n, reps):
    key = np.array(bench.seed_from_u64(SEED), np.uint32)
    out = torch.empty((n, 8), dtype=torch.int32, device="cuda:0")
    for _ in range(3):
        eng.stdrng_random(key, 0, n, 0, flags=DEVICE_PTRS, out=out.data_ptr())
    torch.cuda.synchronize()
    per = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(10):
            eng.stdrng_random(key, 0, n, 0, flags=DEVICE_PTRS, out=out.data_ptr())
        b.record()
        b.synchronize()
        per.append(a.elapsed_time(b) / 10)
    host, _ = eng.stdrng_random(key, 0, 4096, 0)
    assert (out[:4096].cpu().numpy().view(np.uint32) == host).all()
    assert (host == bench.stdrng_nonces(eng, SEED, 4096)).all(), "device draws differ from the host recipe"
    st = stats(per)
    st["draws_per_s"] = round(n / (st["median_ms"] * 1e-3), 1)
    return {"n": n, "what": "sb200_stdrng_random, field 0, SB200_DEVICE_PTRS output; CUDA events over 10 back-to-back calls", **st}


def time_sign(eng, scheme, lg, reps):
    n = 1 << lg
    name = "sign" if scheme == 0 else "sign_double"
    rs = np.random.RandomState(SEED + lg)
    (t_sk, sk), (t_m, msg), (t_nonce, nonce) = pinned((n, 8)), pinned((n, 8)), pinned((n, 8))
    sk[...] = rs.randint(0, 2**32, size=(n, 8), dtype=np.uint64).astype(np.uint32)
    sk[:, 7] &= 0x07FFFFFF
    msg[...] = rs.randint(0, 2**32, size=(n, 8), dtype=np.uint64).astype(np.uint32)
    msg[:, 7] &= 0x3FFFFFFF
    outs = {p: [pinned((n, w)) for w in ((8, 16, 16, 8) if scheme == 1 else (8, 16, 8))] for p in (1, 2)}
    key = np.array(bench.seed_from_u64(SEED), np.uint32)
    lib, h = eng._lib, eng._h

    def path1():
        t0 = time.perf_counter()
        words = [bench.chacha12_blocks(key, lo, min(1 << 20, n - lo)) for lo in range(0, n, 1 << 20)]
        t1 = time.perf_counter()
        for j, lo in enumerate(range(0, n, 1 << 20)):
            nonce[lo:lo + len(words[j])] = eng.scalars_from_wide(words[j].view(np.uint8), 0)
        t2 = time.perf_counter()
        o = outs[1]
        eng.call(name, n, 0, sk.ctypes.data, msg.ctypes.data, nonce.ctypes.data, *[a.ctypes.data for _, a in o])
        t3 = time.perf_counter()
        return (t3 - t0) * 1e3, ((t1 - t0) * 1e3, (t2 - t1) * 1e3, (t3 - t2) * 1e3)

    def path2():
        o = outs[2]
        pos = StdRngPos.of(key, 0)
        t0 = time.perf_counter()
        rc = lib.sb200_sign_stdrng(h, n, 0, scheme, sk.ctypes.data, msg.ctypes.data, None, ctypes.byref(pos),
                                   o[0][1].ctypes.data, o[1][1].ctypes.data, o[2][1].ctypes.data if scheme == 1 else None,
                                   o[-1][1].ctypes.data)
        t1 = time.perf_counter()
        assert rc == 0 and pos.word_pos == 16 * n
        return (t1 - t0) * 1e3

    path1(), path2()  # warm-up: arenas, staging, module loads
    w1, parts, w2 = [], [], []
    for _ in range(reps):  # alternate the two paths
        t, p = path1()
        w1.append(t)
        parts.append(p)
        w2.append(path2())
    same = all((a == b).all() for (_, a), (_, b) in zip(outs[1], outs[2]))
    assert same, f"{name} 2^{lg}: outputs of the two paths differ"
    med = lambda k: round(sorted(p[k] for p in parts)[len(parts) // 2], 3)
    s1, s2 = stats(w1), stats(w2)
    return {"call": name, "n": n, "outputs_byte_identical": same,
            "host_draw": {**s1, "signs_per_s": round(n / (s1["median_ms"] * 1e-3), 1),
                          "parts_median_ms": {"numpy_chacha12": med(0), "scalars_from_wide": med(1), "sign": med(2)}},
            "device_draw": {**s2, "signs_per_s": round(n / (s2["median_ms"] * 1e-3), 1)},
            "speedup_median": round(s1["median_ms"] / s2["median_ms"], 3)}


def typed(lg):
    exe = os.path.join(ROOT, "build", "bench_typed")
    out = subprocess.run([exe, str(lg), "3"], capture_output=True, text=True, timeout=900)
    return json.loads(out.stdout) if out.returncode == 0 else {"error": out.stderr[-400:]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    res = {"card": card()}
    eng = Engine([0])
    try:
        res["a_generation_2_22"] = time_generation(eng, 1 << 22, a.reps)
        print(json.dumps(res["a_generation_2_22"]), flush=True)
        for key, scheme, lg in (("b_sign_2_20", 0, 20), ("b_sign_2_22", 0, 22), ("c_sign_double_2_20", 1, 20)):
            res[key] = time_sign(eng, scheme, lg, a.reps)
            print(json.dumps(res[key]), flush=True)
    finally:
        eng.close()
    earlier = [json.loads(l) for l in open(os.path.join(ROOT, "profiles", "bench_typed_r02b.json")) if l.strip()]
    res["d_e2e_typed"] = {"note": "typed C++ API (tools/bench_typed.cpp), pageable memory; this build against the committed "
                                  "profiles/bench_typed_r02b.json of an earlier build (host-drawn nonces): a comparison across builds",
                          "this_build": [typed(20), typed(22)],
                          "earlier_build": [{k: r[k] for k in ("log2n", "sign_typed_per_s", "sign_typed_ms")} for r in earlier]}
    res["card_after"] = card()
    s = json.dumps(res, indent=1)
    print(s, flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
