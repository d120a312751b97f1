"""What the verifier-side witness rows cost (sb200_verify_witness) next to the calls a prover would otherwise combine.

For each scheme (0 single, 1 double, 2 variable generator) at 2^20 and 2^22 tuples, 10 % of them corrupted (u + 1), in
one process on one GPU, the calls alternated over --reps repetitions (median reported):
  - sb200_verify_witness, SB200_DEVICE_PTRS (inputs and outputs device-resident; CUDA events around one call);
  - sb200_verify_witness from pinned host buffers, end to end (host clock; the call returns when its rows have landed);
  - sb200_verify* (no c_out) and sb200_sign_witness at the same size, device-resident, CUDA events.
Checked in the same run: every verdict equals sb200_verify*'s, the corrupted tuples fail, and the rows of the valid
tuples are bit-identical to sb200_sign_witness's rows of the same signatures.  Each rate is also given as a fraction of
the measured IMAD.WIDE peak (IMAD_PEAK.json), with the per-tuple IMAD.WIDE count of profiles/op_counts.json
(verify_witness_single | _double | _vargen, verify_affine | verify_double_affine | verify_vargen_affine).

Writes DIR/witness_time.json with the card's name and power limit read in the same run.
Usage:  python tools/witness_time.py --out DIR [--reps 5] [--lgs 20,22]     (needs a GPU)"""
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
WIDTH = (11, 19, 13)
VERIFY = ("verify", "verify_double", "verify_vargen")
VERIFY_COUNTS = ("verify_affine", "verify_double_affine", "verify_vargen_affine")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip() or q.stderr.strip()}


def scalars(rs, n, bits):
    a = rs.randint(0, 1 << 32, size=(n, 8), dtype=np.uint64).astype(np.uint32)
    a[:, 7] &= (1 << (bits - 224)) - 1
    return a


def inputs(eng, scheme, n, seed):
    """signed tuples (sign_witness on the device), 10 % with u + 1; the signer's rows; the verify-call inputs"""
    rs = np.random.RandomState(seed)
    sk, nonce, msg = scalars(rs, n, 251), scalars(rs, n, 251), scalars(rs, n, 254)
    gen = eng.keygen(scalars(rs, n, 251)) if scheme == 2 else None
    rows = eng.sign_witness(scheme, sk, msg, nonce, gen=gen, affine=True)
    u = eng.fq_from_mont(np.ascontiguousarray(rows[:, 0]))
    bad = np.zeros(n, bool)
    bad[rs.choice(n, n // 10, replace=False)] = True
    u[bad, 0] ^= 1  # u +- 1 (< r still: u has 251 bits)
    Rr = np.ascontiguousarray(rows[:, 1:3].reshape(n, 16))
    if scheme == 0:
        arrays = [eng.keygen(sk), None, u, Rr, None, msg]
    elif scheme == 1:
        pk, pkp = eng.keygen_double(sk)
        arrays = [pk, pkp, u, Rr, np.ascontiguousarray(rows[:, 3:5].reshape(n, 16)), msg]
    else:
        arrays = [eng.keygen_vargen(sk, gen), gen, u, Rr, None, msg]
    return dict(sign_in=(sk, msg, nonce, gen), rows=rows, bad=bad, arrays=arrays)


def stats(xs):
    s = sorted(xs)
    return {"median_ms": round(s[len(s) // 2], 3), "min_ms": round(s[0], 3), "max_ms": round(s[-1], 3), "reps": len(s)}


def run(eng, scheme, lg, reps, counts, peak):
    n = 1 << lg
    d = inputs(eng, scheme, n, 1000 * scheme + lg)
    lib, h = eng._lib, eng._h
    dev = torch.device("cuda:0")
    to_dev = lambda a: torch.from_numpy(np.ascontiguousarray(a).view(np.int32)).to(dev) if a is not None else None
    P = lambda t: ctypes.c_void_p(t.data_ptr()) if t is not None else None
    di = [to_dev(a) for a in d["arrays"]]
    sk, msg, nonce, gen = (to_dev(a) for a in d["sign_in"])
    bm = torch.zeros((n + 31) // 32, dtype=torch.int32, device=dev)
    bm_v = torch.zeros_like(bm)
    rows = torch.empty((n, WIDTH[scheme] * 8), dtype=torch.int32, device=dev)
    srows = torch.empty_like(rows)
    verify_ins = [x for x in di if x is not None]
    fl = POINTS_AFFINE | DEVICE_PTRS
    calls = {
        "verify_witness_device": lambda: lib.sb200_verify_witness(h, n, fl, scheme, *[P(x) for x in di], P(bm), P(rows)),
        "verify_device": lambda: getattr(lib, "sb200_" + VERIFY[scheme])(h, n, fl, *[P(x) for x in verify_ins], P(bm_v), None),
        "sign_witness_device": lambda: lib.sb200_sign_witness(h, n, (fl if scheme == 2 else DEVICE_PTRS), scheme, P(sk), P(msg),
                                                              P(nonce), P(gen), P(srows)),
    }
    # pinned host buffers for the end-to-end call
    pin = lambda a: (torch.from_numpy(np.ascontiguousarray(a).view(np.int32)).pin_memory() if a is not None else None)
    hi = [pin(a) for a in d["arrays"]]
    hbm = torch.zeros((n + 31) // 32, dtype=torch.int32).pin_memory()
    hrows = torch.empty((n, WIDTH[scheme] * 8), dtype=torch.int32).pin_memory()
    calls["verify_witness_pinned_e2e"] = lambda: lib.sb200_verify_witness(h, n, POINTS_AFFINE, scheme, *[P(x) for x in hi], P(hbm),
                                                                          P(hrows))
    for name, fn in calls.items():  # warm-up of every shape, and the return codes
        assert fn() == 0, name
    torch.cuda.synchronize()
    times = {k: [] for k in calls}
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
    # outputs of the last repetition
    unpack = lambda t: np.unpackbits(t.cpu().numpy().view(np.uint8), bitorder="little")[:n].astype(bool)
    ok, ok_v, ok_h = unpack(bm), unpack(bm_v), unpack(hbm)
    got, got_h = rows.cpu().numpy().view(np.uint32).reshape(n, -1, 8), hrows.numpy().view(np.uint32).reshape(n, -1, 8)
    signer = d["rows"]
    assert (ok == ok_v).all() and (ok_h == ok).all(), "verdicts differ from sb200_verify*"
    assert (ok == ~d["bad"]).all(), "a corrupted tuple passed or a signed one failed"
    assert (got[ok] == signer[ok]).all() and (got_h == got).all(), "rows of valid tuples differ from sign_witness's"
    assert (srows.cpu().numpy().view(np.uint32).reshape(n, -1, 8) == signer).all()
    out = {"scheme": NAMES[scheme], "n": n, "corrupted": int(d["bad"].sum()), "checks": "verdicts == sb200_verify*, rows of valid tuples == sign_witness rows"}
    wkey, vkey = "verify_witness_" + NAMES[scheme], VERIFY_COUNTS[scheme]
    for name, xs in times.items():
        st = stats(xs)
        st["tuples_per_s"] = round(n / (st["median_ms"] * 1e-3), 1)
        key = {"verify_device": vkey, "sign_witness_device": None}.get(name, wkey)
        if key:
            st["imad_wide_per_tuple"] = counts[key]["imad_wide_per_tuple"]
            st["frac_of_imad_peak"] = round(st["tuples_per_s"] * counts[key]["imad_wide_per_tuple"] / peak, 4)
        out[name] = st
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--lgs", default="20,22")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("witness_time.py needs a GPU")
    counts = json.load(open(os.path.join(ROOT, "profiles", "op_counts.json")))
    peak = json.load(open(os.path.join(ROOT, "IMAD_PEAK.json")))["imad_wide_per_s"]
    res = {"card": card(), "imad_peak_per_s": peak, "runs": []}
    eng = Engine([0])
    try:
        for lg in (int(x) for x in args.lgs.split(",")):
            for scheme in range(3):
                r = run(eng, scheme, lg, args.reps, counts, peak)
                print(json.dumps(r), flush=True)
                res["runs"].append(r)
                torch.cuda.empty_cache()
    finally:
        eng.close()
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "witness_time.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res["card"]))


if __name__ == "__main__":
    main()
