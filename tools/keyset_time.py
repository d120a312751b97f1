"""What verification against registered keys (include/schnorr_b200_keyset.h) costs and saves, next to sb200_verify*.

In one process on one GPU, for each scheme (0 single, 1 double, 2 variable generator):
  - the keyset build (sb200_keyset_create from device-resident keys, to return) for 2^10, 2^14 and 2^16 keys;
  - for K = 2^8, 2^12 and 2^16 keys, 2^22 tuples signed by keys drawn uniformly, 10 % corrupted (u + 1, m + 1, R + B, a
    neighbour's key index), verified by sb200_verify_keyset and by sb200_verify* on the gathered keys:
      device-resident (SB200_DEVICE_PTRS, CUDA events around one call) and from pinned host buffers (host clock, the call
      returns when its results have landed);
    the four calls alternated over --reps repetitions (medians reported), verdicts and challenges of the two calls
    compared in every repetition;
  - the break-even: signatures per key above which build + keyset verification beats sb200_verify* (device-resident).
Writes DIR/keyset_time.json with the card's name and power limit read in the same run.
Usage:  python tools/keyset_time.py --out DIR [--reps 5] [--lg 22]     (needs a GPU)"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT]
sys.dont_write_bytecode = True
import numpy as np  # noqa: E402
import torch  # noqa: E402

from schnorr_b200 import Engine  # noqa: E402
from schnorr_b200._lib import DEVICE_PTRS, POINTS_AFFINE  # noqa: E402

NAMES = ("single", "double", "vargen")
VERIFY = ("verify", "verify_double", "verify_vargen")
COUNTS = (("verify_affine", "keyset_verify_single"), ("verify_double_affine", "keyset_verify_double"),
          ("verify_vargen_affine", "keyset_verify_vargen"))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip() or q.stderr.strip()}


def scalars(rs, n, bits):
    a = rs.randint(0, 1 << 32, size=(n, 8), dtype=np.uint64).astype(np.uint32)
    a[:, 7] &= (1 << (bits - 224)) - 1
    return a


def stats(xs):
    s = sorted(xs)
    return {"median_ms": round(s[len(s) // 2], 3), "min_ms": round(s[0], 3), "max_ms": round(s[-1], 3), "reps": len(s)}


def keys_of(eng, scheme, K, rs):
    sk = scalars(rs, K, 251)
    if scheme == 0:
        return sk, eng.keygen(sk), None
    if scheme == 1:
        return (sk,) + eng.keygen_double(sk)
    gen = eng.keygen(scalars(rs, K, 251))
    return sk, eng.keygen_vargen(sk, gen), gen


def create(eng, scheme, pk, pk2):
    """sb200_keyset_create from device-resident keys: (handle, seconds to return)"""
    h = ctypes.c_void_p()
    P = lambda t: ctypes.c_void_p(t.data_ptr()) if t is not None else None
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    rc = eng._lib.sb200_keyset_create(eng._h, scheme, pk.shape[0], POINTS_AFFINE | DEVICE_PTRS, P(pk), P(pk2), None, ctypes.byref(h))
    dt = time.perf_counter() - t0
    assert rc == 0, rc
    return h, dt


def build_times(eng, scheme, reps):
    out = {}
    for lgk in (10, 14, 16):
        K = 1 << lgk
        _, pk, pk2 = keys_of(eng, scheme, K, np.random.RandomState(lgk))
        dev = lambda a: torch.from_numpy(a.view(np.int32)).cuda() if a is not None else None
        pkd, pk2d = dev(pk), dev(pk2)
        xs = []
        for _ in range(reps):
            h, dt = create(eng, scheme, pkd, pk2d)
            eng._lib.sb200_keyset_destroy(h)
            xs.append(dt * 1e3)
        st = stats(xs)
        st["us_per_key"] = round(st["median_ms"] * 1e3 / K, 3)
        st["table_bytes_per_device"] = K * (1 if scheme == 0 else 2) * 396288
        out[f"2^{lgk}"] = st
    return out


def tuples(eng, scheme, sk, pk, pk2, n, rs):
    """n tuples over the keys, key index uniform; 10 % corrupted: u + 1, m + 1, R + B, a neighbour's key index"""
    K = sk.shape[0]
    idx = rs.randint(0, K, size=n).astype(np.uint32)
    nonce, m = scalars(rs, n, 251), scalars(rs, n, 254)
    Rp = None
    if scheme == 0:
        u, Rr, _ = eng.sign(sk[idx], m, nonce)
    elif scheme == 1:
        u, Rr, Rp, _ = eng.sign_double(sk[idx], m, nonce)
    else:
        u, Rr, _ = eng.sign_vargen(sk[idx], pk2[idx], m, nonce)
    cat = np.full(n, -1)
    bad = rs.choice(n, n // 10, replace=False)
    cat[bad] = rs.randint(0, 4, size=len(bad))
    i = np.nonzero(cat == 0)[0]
    u[i, 0] ^= 1  # u +- 1 (still < r)
    i = np.nonzero(cat == 1)[0]
    m[i, 0] ^= 1
    i = np.nonzero(cat == 2)[0]  # R + B = (nonce + 1) B
    n1 = nonce[i].copy()
    n1[:, 0] += 1  # nonce < 2^251 with a random low word: no carry out of it but with probability 2^-32 ...
    assert (n1[:, 0] != 0).all()  # ... which this run did not meet
    Rr[i] = eng.keygen(n1) if scheme != 2 else eng.keygen_vargen(n1, pk2[idx[i]])
    i = np.nonzero(cat == 3)[0]
    idx[i] = (idx[i] + 1) % K
    return idx, u, Rr, Rp, m, cat


def run(eng, scheme, lgk, n, reps, counts):
    rs = np.random.RandomState(100 * scheme + lgk)
    K = 1 << lgk
    sk, pk, pk2 = keys_of(eng, scheme, K, rs)
    idx, u, Rr, Rp, m, cat = tuples(eng, scheme, sk, pk, pk2, n, rs)
    gathered = [pk[idx]] + ([pk2[idx]] if scheme else []) + [u, Rr] + ([Rp] if scheme == 1 else []) + [m]
    ks_in = [idx, u, Rr, Rp if scheme == 1 else None, m]
    lib, h = eng._lib, eng._h
    P = lambda t: ctypes.c_void_p(t.data_ptr()) if t is not None else None
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a).view(np.int32)).cuda() if a is not None else None
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a).view(np.int32)).pin_memory() if a is not None else None
    kh, build_s = create(eng, scheme, dev(pk), dev(pk2))
    try:
        outs = {}

        def call(name, ks_call, arrays, flags, on_dev):
            bm = (torch.zeros if on_dev else lambda *a, **k: torch.zeros(*a, **k).pin_memory())((n + 31) // 32, dtype=torch.int32,
                                                                                                   **({"device": "cuda"} if on_dev else {}))
            c = torch.zeros((n, 8), dtype=torch.int32, device="cuda") if on_dev else torch.zeros((n, 8), dtype=torch.int32).pin_memory()
            outs[name] = (bm, c)
            if ks_call:
                return lambda: lib.sb200_verify_keyset(h, kh, n, flags, *[P(x) for x in arrays], P(bm), P(c))
            return lambda: getattr(lib, "sb200_" + VERIFY[scheme])(h, n, flags, *[P(x) for x in arrays], P(bm), P(c))

        fl = POINTS_AFFINE
        calls = {
            "keyset_device": call("keyset_device", True, [dev(x) for x in ks_in], fl | DEVICE_PTRS, True),
            "verify_device": call("verify_device", False, [dev(x) for x in gathered], fl | DEVICE_PTRS, True),
            "keyset_pinned_e2e": call("keyset_pinned_e2e", True, [pin(x) for x in ks_in], fl, False),
            "verify_pinned_e2e": call("verify_pinned_e2e", False, [pin(x) for x in gathered], fl, False),
        }
        for name, fn in calls.items():  # warm-up of every shape, and the return codes
            assert fn() == 0, name
        torch.cuda.synchronize()
        times = {k: [] for k in calls}
        unpack = lambda t: np.unpackbits(t.cpu().numpy().view(np.uint8), bitorder="little")[:n].astype(bool)
        for _ in range(reps):
            for name, fn in calls.items():
                if name.endswith("e2e"):
                    t0 = time.perf_counter()
                    assert fn() == 0
                    times[name].append((time.perf_counter() - t0) * 1e3)
                else:
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a.record()
                    assert fn() == 0
                    b.record()
                    b.synchronize()
                    times[name].append(a.elapsed_time(b))
            ref_ok, ref_c = unpack(outs["verify_device"][0]), outs["verify_device"][1].cpu().numpy()
            for name in calls:  # every repetition: verdicts and challenges of all four calls agree
                assert (unpack(outs[name][0]) == ref_ok).all(), name
                assert (outs[name][1].cpu().numpy() == ref_c).all(), name
        assert ref_ok[cat == -1].all() and not ref_ok[cat >= 0].any(), "a signed tuple failed or a corrupted one passed"
    finally:
        lib.sb200_keyset_destroy(kh)
    res = {"scheme": NAMES[scheme], "n": n, "keys": K, "corrupted": int((cat >= 0).sum()),
           "checks": "verdicts and c_out of sb200_verify_keyset == sb200_verify* on the gathered keys, every repetition",
           "build_ms_in_this_run": round(build_s * 1e3, 3)}
    for name, xs in times.items():
        st = stats(xs)
        st["tuples_per_s"] = round(n / (st["median_ms"] * 1e-3), 1)
        st["imad_wide_per_tuple"] = counts[COUNTS[scheme][name.startswith("keyset")]]["imad_wide_per_tuple"]
        res[name] = st
    res["speedup_device"] = round(res["verify_device"]["median_ms"] / res["keyset_device"]["median_ms"], 3)
    res["speedup_pinned_e2e"] = round(res["verify_pinned_e2e"]["median_ms"] / res["keyset_pinned_e2e"]["median_ms"], 3)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--lg", type=int, default=22)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("keyset_time.py needs a GPU")
    counts = json.load(open(os.path.join(ROOT, "profiles", "op_counts.json")))
    res = {"card": card(), "n": 1 << args.lg, "builds": {}, "runs": [], "break_even_signatures_per_key": {}}
    eng = Engine([0])
    try:
        for scheme in range(3):
            res["builds"][NAMES[scheme]] = b = build_times(eng, scheme, 3)
            print(json.dumps({NAMES[scheme]: b}), flush=True)
            for lgk in (8, 12, 16):
                r = run(eng, scheme, lgk, 1 << args.lg, args.reps, counts)
                print(json.dumps(r), flush=True)
                res["runs"].append(r)
                torch.cuda.empty_cache()
                # build(K) + K s t_keyset < K s t_verify  <=>  s > build(K) / (K (t_verify - t_keyset)), per-tuple times
                saved = (r["verify_device"]["median_ms"] - r["keyset_device"]["median_ms"]) / r["n"]
                bk = b.get(f"2^{lgk}", {}).get("median_ms", r["build_ms_in_this_run"])
                res["break_even_signatures_per_key"][f"{NAMES[scheme]} K=2^{lgk}"] = (
                    round(bk / ((1 << lgk) * saved), 2) if saved > 0 else None)
    finally:
        eng.close()
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "keyset_time.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"card": res["card"], "break_even": res["break_even_signatures_per_key"]}))


if __name__ == "__main__":
    main()
