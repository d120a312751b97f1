"""What the byte-level keyset verification and the live keyset updates (include/schnorr_b200_keyset_live.h) cost.

In one process on one GPU, for each scheme (0 single, 1 double, 2 variable generator):
  - for K = 2^12 and 2^16 keys registered from their to_bytes() form (sb200_keyset_create_bytes), 2^22 tuples signed by
    keys drawn uniformly, 10 % corrupted (u + 1, m + 1, R + B, a neighbour's key index), as wire bytes, verified by
      sb200_verify_keyset_bytes   device-resident (SB200_DEVICE_PTRS, CUDA events around one call) and from pinned host
                                  buffers (host clock: the call returns when its results have landed),
      sb200_verify_keyset         device-resident, on the same tuples as limbs,
      sb200_verify*_bytes         device-resident, on the gathered key bytes;
    the calls alternated over --reps repetitions (medians reported), the verdicts of all paths compared in every
    repetition.  decode_ms = byte-level keyset call - limb keyset call: the decode launch and its scratch round trip.
  - on a keyset of 2^16 keys: sb200_keyset_update of m = 1, 64 and 2048 scattered slots (keys in host memory, to return),
    sb200_keyset_revoke of 2048 slots, and sb200_keyset_create of all 2^16 keys from device-resident limbs.
Writes DIR/keyset_live_time.json with the card's name and power limit read in the same run.
Usage:  python tools/keyset_live_time.py --out DIR [--reps 5] [--lg 22]     (needs a GPU)"""
import argparse
import ctypes
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tools")]
sys.dont_write_bytecode = True
import numpy as np  # noqa: E402
import torch  # noqa: E402

from keyset_time import card, create, keys_of, stats, tuples  # noqa: E402
from schnorr_b200 import Engine  # noqa: E402
from schnorr_b200._lib import DEVICE_PTRS, POINTS_AFFINE, aligned_empty  # noqa: E402

NAMES = ("single", "double", "vargen")
VERIFY_BYTES = ("verify_bytes", "verify_double_bytes", "verify_vargen_bytes")


def key_bytes(eng, pk, pk2):
    b = eng.points_compress(pk)
    return b if pk2 is None else np.ascontiguousarray(np.concatenate([b, eng.points_compress(pk2)], axis=1))


def wire(eng, u, Rr, Rp, m):
    n = u.shape[0]
    parts = [np.ascontiguousarray(u).view(np.uint8).reshape(n, 32), eng.points_compress(Rr)]
    if Rp is not None:
        parts.append(eng.points_compress(Rp))
    return np.ascontiguousarray(np.concatenate(parts, axis=1)), np.ascontiguousarray(eng.fq_from_mont(m).view(np.uint8).reshape(n, 32))


P = lambda t: ctypes.c_void_p(t.data_ptr()) if t is not None else None
dev = lambda a: torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1)).cuda() if a is not None else None
devk = lambda a: torch.from_numpy(np.ascontiguousarray(a).view(np.int32)).cuda() if a is not None else None  # [K, 16] rows
pin = lambda a: torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1)).pin_memory() if a is not None else None


def aligned(a):
    if a is None:
        return None
    b = aligned_empty(a.shape, a.dtype)
    b[...] = a
    return b


def run(eng, scheme, lgk, n, reps):
    rs = np.random.RandomState(100 * scheme + lgk + 7)
    K = 1 << lgk
    sk, pk, pk2 = keys_of(eng, scheme, K, rs)
    idx, u, Rr, Rp, m, cat = tuples(eng, scheme, sk, pk, pk2, n, rs)
    pkb = key_bytes(eng, pk, pk2)
    sig, msg = wire(eng, u, Rr, Rp, m)
    lib, h = eng._lib, eng._h
    kb = ctypes.c_void_p()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    keys_d = [dev(pkb), devk(pk), devk(pk2)]  # alive until the builds have returned
    assert lib.sb200_keyset_create_bytes(h, scheme, K, DEVICE_PTRS, P(keys_d[0]), None, ctypes.byref(kb)) == 0
    create_bytes_ms = (time.perf_counter() - t0) * 1e3
    kl, _ = create(eng, scheme, keys_d[1], keys_d[2])
    outs = {}

    def bitmaps(name, on_dev, with_inv):
        mk = (lambda: torch.zeros((n + 31) // 32, dtype=torch.int32, device="cuda")) if on_dev else \
            (lambda: torch.zeros((n + 31) // 32, dtype=torch.int32).pin_memory())
        outs[name] = (mk(), mk() if with_inv else None)
        return outs[name]

    try:
        ksb_d = [dev(idx), dev(sig), dev(msg)]
        ksb_p = [pin(idx), pin(sig), pin(msg)]
        lim_d = [dev(idx), dev(u), dev(Rr), dev(Rp), dev(m)]
        vb_d = [dev(pkb[idx]), ksb_d[1], ksb_d[2]]
        calls = {}
        bm, iv = bitmaps("keyset_bytes_device", True, True)
        calls["keyset_bytes_device"] = lambda bm=bm, iv=iv: lib.sb200_verify_keyset_bytes(h, kb, n, DEVICE_PTRS, *map(P, ksb_d), P(bm), P(iv))
        bm, iv = bitmaps("keyset_bytes_pinned_e2e", False, True)
        calls["keyset_bytes_pinned_e2e"] = lambda bm=bm, iv=iv: lib.sb200_verify_keyset_bytes(h, kb, n, 0, *map(P, ksb_p), P(bm), P(iv))
        bm, _ = bitmaps("keyset_device", True, False)
        calls["keyset_device"] = lambda bm=bm: lib.sb200_verify_keyset(h, kl, n, POINTS_AFFINE | DEVICE_PTRS, *map(P, lim_d), P(bm), None)
        bm, iv = bitmaps("verify_bytes_device", True, True)
        calls["verify_bytes_device"] = lambda bm=bm, iv=iv: getattr(lib, "sb200_" + VERIFY_BYTES[scheme])(h, n, DEVICE_PTRS, *map(P, vb_d), P(bm), P(iv))
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
            ref = unpack(outs["verify_bytes_device"][0])
            for name in calls:  # every repetition: the verdicts of all paths agree, and nothing was reported undecodable
                assert (unpack(outs[name][0]) == ref).all(), name
                if outs[name][1] is not None:
                    assert not unpack(outs[name][1]).any(), name
        assert ref[cat == -1].all() and not ref[cat >= 0].any(), "a signed tuple failed or a corrupted one passed"
    finally:
        lib.sb200_keyset_destroy(kb)
        lib.sb200_keyset_destroy(kl)
    res = {"scheme": NAMES[scheme], "n": n, "keys": K, "corrupted": int((cat >= 0).sum()),
           "checks": "verdicts of sb200_verify_keyset_bytes (device, pinned) == sb200_verify_keyset == sb200_verify*_bytes on "
                     "the gathered key bytes, every repetition; no tuple reported undecodable",
           "create_bytes_ms_in_this_run": round(create_bytes_ms, 3)}
    for name, xs in times.items():
        st = stats(xs)
        st["tuples_per_s"] = round(n / (st["median_ms"] * 1e-3), 1)
        res[name] = st
    res["decode_ms"] = round(res["keyset_bytes_device"]["median_ms"] - res["keyset_device"]["median_ms"], 3)
    res["speedup_vs_verify_bytes_device"] = round(res["verify_bytes_device"]["median_ms"] / res["keyset_bytes_device"]["median_ms"], 3)
    return res


def live(eng, scheme, reps):
    """update of m slots, revoke of 2048 slots and a full create, on 2^16 keys"""
    K = 1 << 16
    rs = np.random.RandomState(900 + scheme)
    sk, pk, pk2 = keys_of(eng, scheme, K, rs)
    _, npk, npk2 = keys_of(eng, scheme, 2048, rs)
    pkd, pk2d = devk(pk), devk(pk2)
    out = {"keys": K}
    xs = []
    for _ in range(3):
        h, dt = create(eng, scheme, pkd, pk2d)
        eng._lib.sb200_keyset_destroy(h)
        xs.append(dt * 1e3)
    out["create_2^16"] = stats(xs)
    h, _ = create(eng, scheme, pkd, pk2d)
    try:
        for mm in (1, 64, 2048):
            xs = []
            for r in range(reps):
                slots = aligned(rs.choice(K, mm, replace=False).astype(np.uint32))
                a, a2 = aligned(npk[:mm]), aligned(npk2[:mm] if npk2 is not None else None)
                okw = np.zeros((mm + 31) // 32 + 1, np.uint32)
                t0 = time.perf_counter()
                rc = eng._lib.sb200_keyset_update(h, mm, POINTS_AFFINE, slots.ctypes.data, a.ctypes.data,
                                                  a2.ctypes.data if a2 is not None else None, okw.ctypes.data)
                xs.append((time.perf_counter() - t0) * 1e3)
                assert rc == 0 and np.unpackbits(okw.view(np.uint8), bitorder="little")[:mm].all()
            out[f"update_m={mm}"] = stats(xs)
        xs = []
        for r in range(reps):
            slots = aligned(rs.choice(K, 2048, replace=False).astype(np.uint32))
            t0 = time.perf_counter()
            assert eng._lib.sb200_keyset_revoke(h, 2048, slots.ctypes.data) == 0
            xs.append((time.perf_counter() - t0) * 1e3)
        out["revoke_m=2048"] = stats(xs)
    finally:
        eng._lib.sb200_keyset_destroy(h)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--lg", type=int, default=22)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("keyset_live_time.py needs a GPU")
    res = {"card": card(), "n": 1 << args.lg, "runs": [], "live": {}}
    eng = Engine([0])
    try:
        for scheme in range(3):
            for lgk in (12, 16):
                r = run(eng, scheme, lgk, 1 << args.lg, args.reps)
                print(json.dumps(r), flush=True)
                res["runs"].append(r)
                torch.cuda.empty_cache()
            res["live"][NAMES[scheme]] = lv = live(eng, scheme, args.reps)
            print(json.dumps({NAMES[scheme]: lv}), flush=True)
            torch.cuda.empty_cache()
    finally:
        eng.close()
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "keyset_live_time.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"card": res["card"]}))


if __name__ == "__main__":
    main()
