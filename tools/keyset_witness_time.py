"""What witness rows against a keyset (include/schnorr_b200_keyset_witness.h) cost, next to sb200_verify_witness and
sb200_verify_keyset.

In one process on one GPU, for each scheme (0 single, 1 double, 2 variable generator) and K = 2^12 and 2^16 keys: 2^22
tuples signed by keys drawn uniformly, 10 % corrupted (u + 1, m + 1, R + B, a neighbour's key index), run through
  - sb200_verify_witness_keyset (limbs) and sb200_verify_witness_keyset_bytes (sig64 / sig96 and canonical messages),
  - sb200_verify_witness on the gathered keys,
  - sb200_verify_keyset (verdicts only),
each device-resident (SB200_DEVICE_PTRS, CUDA events around one call) and from pinned host buffers (host clock, the call
returns when its results have landed).  The eight calls alternate over --reps repetitions (medians reported); in every
repetition the rows of the three witness calls and the verdicts of all four are compared on the device.  The pinned
figures include copying the rows (352 / 608 / 416 B per tuple) back to host memory, so they can be bound by that copy.
`--quick`: device-resident sb200_verify_witness_keyset only, K = 2^12, for timing library variants (SB200_LIB) against
each other in alternated processes.
Writes DIR/keyset_witness_time.json with the card's name and power limit read in the same run.
Usage:  python tools/keyset_witness_time.py --out DIR [--reps 5] [--lg 22] [--quick]     (needs a GPU)"""
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
from schnorr_b200._lib import DEVICE_PTRS, LIB_PATH, POINTS_AFFINE  # noqa: E402

NAMES = ("single", "double", "vargen")
WIDTH = (11, 19, 13)
COUNTS = {"witness_keyset": ("keyset_witness_single", "keyset_witness_double", "keyset_witness_vargen"),
          "witness": ("verify_witness_single", "verify_witness_double", "verify_witness_vargen"),
          "keyset": ("keyset_verify_single", "keyset_verify_double", "keyset_verify_vargen")}


DUMP = None  # where mismatch() leaves the first differing tuples


def mismatch(name, bm, rows, ref_bm, ref_rows, idx, u, Rr, Rp, m, cat, pk, pk2):
    """write the first differing tuples (inputs, both rows) to DUMP, then fail"""
    n = len(idx)
    ub = lambda t: np.unpackbits(t.cpu().numpy().view(np.uint8), bitorder="little")[:n].astype(bool)
    d = ub(bm) != ub(ref_bm)
    if rows is not None:
        d |= (rows.cuda() != ref_rows).any(dim=1).cpu().numpy()
    i = np.nonzero(d)[0]
    sel = i[:256]
    os.makedirs(DUMP, exist_ok=True)
    np.savez(os.path.join(DUMP, f"mismatch_{name}.npz"), i=sel, count=len(i), idx=idx[sel], key_pk=pk[idx[sel]],
             key_pk2=pk2[idx[sel]] if pk2 is not None else np.zeros(0), u=u[sel], R=Rr[sel], Rp=Rp[sel] if Rp is not None else np.zeros(0),
             m=m[sel], cat=cat[sel], ok=ub(bm)[sel], ref_ok=ub(ref_bm)[sel],
             rows=rows[torch.from_numpy(sel).cuda()].cpu().numpy() if rows is not None else np.zeros(0),
             ref_rows=ref_rows[torch.from_numpy(sel).cuda()].cpu().numpy())
    raise AssertionError(f"{name}: {len(i)} tuples differ from the reference, first {sel[:8].tolist()}")


def run(eng, scheme, lgk, n, reps, counts, quick=False):
    rs = np.random.RandomState(100 * scheme + lgk)
    K = 1 << lgk
    sk, pk, pk2 = keys_of(eng, scheme, K, rs)
    idx, u, Rr, Rp, m, cat = tuples(eng, scheme, sk, pk, pk2, n, rs)
    gathered = [pk[idx]] + ([pk2[idx]] if scheme else []) + [u, Rr] + ([Rp] if scheme == 1 else []) + [m]
    ks_in = [idx, u, Rr, Rp if scheme == 1 else None, m]
    sig = np.concatenate([u.view(np.uint8).reshape(n, 32), eng.points_compress(Rr)] +
                         ([eng.points_compress(Rp)] if scheme == 1 else []), axis=1)
    msg = eng.fq_from_mont(m).view(np.uint8).reshape(n, 32)
    by_in = [idx, sig, msg]
    lib, h = eng._lib, eng._h
    P = lambda t: ctypes.c_void_p(t.data_ptr()) if t is not None else None
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a).view(np.int32)).cuda() if a is not None else None
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a).view(np.int32)).pin_memory() if a is not None else None
    kh, _ = create(eng, scheme, dev(pk), dev(pk2))
    W = 8 * WIDTH[scheme]
    try:
        outs, held = {}, []

        def call(name, what, arrays, flags, on_dev):
            z = (lambda *s: torch.zeros(*s, dtype=torch.int32, device="cuda")) if on_dev else \
                (lambda *s: torch.zeros(*s, dtype=torch.int32).pin_memory())
            bm, rows = z((n + 31) // 32), (z(n, W) if what != "keyset" else None)
            outs[name] = (bm, rows)
            held.append(arrays)  # the input tensors live as long as the calls that read them
            a = [P(x) for x in arrays]
            if what == "witness_keyset":
                return lambda: lib.sb200_verify_witness_keyset(h, kh, n, flags, *a, P(bm), P(rows))
            if what == "witness_keyset_bytes":
                return lambda: lib.sb200_verify_witness_keyset_bytes(h, kh, n, flags, *a, P(bm), P(rows), None)
            if what == "witness":
                if scheme == 0:
                    a = a[:1] + [None] + a[1:3] + [None] + a[3:]
                elif scheme == 2:
                    a = a[:4] + [None] + a[4:]
                return lambda: lib.sb200_verify_witness(h, n, flags, scheme, *a, P(bm), P(rows))
            return lambda: lib.sb200_verify_keyset(h, kh, n, flags, *a, P(bm), None)

        fl = POINTS_AFFINE
        calls = {"witness_keyset_device": call("witness_keyset_device", "witness_keyset", [dev(x) for x in ks_in], fl | DEVICE_PTRS, True)}
        if not quick:
            calls.update({
                "witness_keyset_bytes_device": call("witness_keyset_bytes_device", "witness_keyset_bytes", [dev(x) for x in by_in],
                                                    DEVICE_PTRS, True),
                "witness_device": call("witness_device", "witness", [dev(x) for x in gathered], fl | DEVICE_PTRS, True),
                "keyset_device": call("keyset_device", "keyset", [dev(x) for x in ks_in], fl | DEVICE_PTRS, True),
                "witness_keyset_pinned_e2e": call("witness_keyset_pinned_e2e", "witness_keyset", [pin(x) for x in ks_in], fl, False),
                "witness_keyset_bytes_pinned_e2e": call("witness_keyset_bytes_pinned_e2e", "witness_keyset_bytes", [pin(x) for x in by_in],
                                                        0, False),
                "witness_pinned_e2e": call("witness_pinned_e2e", "witness", [pin(x) for x in gathered], fl, False),
                "keyset_pinned_e2e": call("keyset_pinned_e2e", "keyset", [pin(x) for x in ks_in], fl, False),
            })
        for name, fn in calls.items():  # warm-up of every shape, and the return codes
            assert fn() == 0, name
        torch.cuda.synchronize()
        times = {k: [] for k in calls}
        ref = "witness_device" if not quick else "witness_keyset_device"
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
            ref_bm, ref_rows = outs[ref]
            for name in calls:  # every repetition: the rows of the witness calls and the verdicts of all calls agree
                bm, rows = outs[name]
                if not torch.equal(bm.cuda(), ref_bm) or (rows is not None and not torch.equal(rows.cuda(), ref_rows)):
                    mismatch(name, bm, rows, ref_bm, ref_rows, idx, u, Rr, Rp, m, cat, pk, pk2)
        ok = np.unpackbits(outs[ref][0].cpu().numpy().view(np.uint8), bitorder="little")[:n].astype(bool)
        assert ok[cat == -1].all() and not ok[cat >= 0].any(), "a signed tuple failed or a corrupted one passed"
    finally:
        lib.sb200_keyset_destroy(kh)
    res = {"scheme": NAMES[scheme], "n": n, "keys": K, "corrupted": int((cat >= 0).sum()), "row_bytes": 4 * W,
           "checks": "rows and verdicts of sb200_verify_witness_keyset, _bytes and sb200_verify_witness on the gathered keys "
                     "equal, and verdicts of sb200_verify_keyset equal, every repetition" if not quick else "repetitions equal"}
    for name, xs in times.items():
        st = stats(xs)
        st["tuples_per_s"] = round(n / (st["median_ms"] * 1e-3), 1)
        kind = "witness_keyset" if name.startswith("witness_keyset") else "witness" if name.startswith("witness") else "keyset"
        st["imad_wide_per_tuple"] = counts[COUNTS[kind][scheme]]["imad_wide_per_tuple"]
        res[name] = st
    if not quick:
        for sfx in ("device", "pinned_e2e"):
            res[f"speedup_vs_witness_{sfx}"] = round(res[f"witness_{sfx}"]["median_ms"] / res[f"witness_keyset_{sfx}"]["median_ms"], 3)
            res[f"cost_vs_keyset_verify_{sfx}"] = round(res[f"witness_keyset_{sfx}"]["median_ms"] / res[f"keyset_{sfx}"]["median_ms"], 3)
        res["row_bytes_per_s_pinned_e2e"] = round(res["witness_keyset_pinned_e2e"]["tuples_per_s"] * 4 * W / 1e9, 2)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--lg", type=int, default=22)
    ap.add_argument("--quick", action="store_true")
    args = ap.parse_args()
    global DUMP
    DUMP = args.out
    if not torch.cuda.is_available():
        sys.exit("keyset_witness_time.py needs a GPU")
    counts = json.load(open(os.path.join(ROOT, "profiles", "op_counts.json")))
    res = {"card": card(), "library": os.path.relpath(LIB_PATH, ROOT), "n": 1 << args.lg, "runs": []}
    eng = Engine([0])
    try:
        for scheme in range(3):
            for lgk in ((12,) if args.quick else (12, 16)):
                r = run(eng, scheme, lgk, 1 << args.lg, args.reps, counts, args.quick)
                print(json.dumps(r), flush=True)
                res["runs"].append(r)
                torch.cuda.empty_cache()
    finally:
        eng.close()
    os.makedirs(args.out, exist_ok=True)
    name = "keyset_witness_time_quick.json" if args.quick else "keyset_witness_time.json"
    with open(os.path.join(args.out, name), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"card": res["card"], "library": res["library"]}))


if __name__ == "__main__":
    main()
