"""Count the field operations / 32x32 limb products one tuple costs in each kernel, by running the
instrumented HOST build of the very same per-tuple code (tests/host_witness.cpp = tests/host_arith.cpp + the
verifier-side witness rows).  Writes
profiles/op_counts.json, which bench.py's roofline uses as "work per tuple"."""
import json, os, sys, random
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "tests"), os.path.join(ROOT, "oracle")]
import numpy as np
import hostlib as H, schnorr_oracle as o, vectors as V

# Host build with the DEVICE's comb width (16-bit windows).  Building the whole 50 MB table with the emulated
# arithmetic would take hours, so only the entries the measured scalars touch are filled in (from the oracle).
import ctypes, subprocess
so16 = os.path.join(ROOT, "build", "host_arith16.so")
subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-DSB_COMB_BITS=16", "-include",
                       os.path.join(ROOT, "tests", "host_shim.h"), "-o", so16, os.path.join(ROOT, "tests", "host_witness.cpp")])
lib = ctypes.CDLL(so16)
H.setup_hades(lib)  # Hades tables derived from the oracle's current round constants, as sb200_init_ex does
W, NWIN, NENT = 16, 16, (1 << 15) + 1
tab = [np.zeros(NWIN * NENT * 24, np.uint32), np.zeros(NWIN * NENT * 24, np.uint32)]
for t in tab:  # entry 0 of every window = identity (1, 1, 0)
    for j in range(NWIN):
        t[(j * NENT) * 24:(j * NENT) * 24 + 16] = np.concatenate([H.mont(1), H.mont(1)])

def fill(k):
    kp = k + int("8000" * 16, 16)
    for j in range(NWIN):
        d = ((kp >> (16 * j)) & 0xFFFF) - 32768
        e = abs(d)
        if e == 0: continue
        for t, B in zip(tab, (o.G, o.G_NUMS)):
            x, y = V.mul(B, e << (16 * j))
            off = (j * NENT + e) * 24
            t[off:off + 24] = np.concatenate([H.mont((y + x) % o.Q), H.mont((y - x) % o.Q), H.mont(2 * o.D * x * y % o.Q)])

rnd = random.Random(3)
sk, nonce, m = rnd.randrange(o.R), rnd.randrange(o.R), rnd.randrange(o.Q)
fill(nonce)
u, Rp, c = o.sign(sk, nonce, m, mul=V.mul)
pk = V.mul(o.G, sk)
fill(u)
fill(o.sign_double(sk, nonce, m, mul=V.mul)[0])
cnt = np.zeros(10, np.uint64)
buf = np.zeros(8, np.uint32)

def measure(fn, lib=lib):
    lib.h_counts_reset(); fn(); lib.h_counts_get(H.ptr(cnt))
    w, mul, sqr, addsub, frm, dot5, dfma = (int(x) for x in cnt[:7])
    return {"imad_wide_per_tuple": w, "fq_mul": mul, "fq_sqr": sqr, "fq_dot5": dot5, "fq_addsub": addsub, "fr_mont_mul": frm, "dfma": dfma}

out = {}
z1, z2 = rnd.randrange(1, o.Q), rnd.randrange(1, o.Q)
out["verify_affine"] = measure(lambda: lib.h_verify(H.ptr(H.pt_mont(pk)), H.ptr(H.limbs(u)), H.ptr(H.pt_mont(Rp)), H.ptr(H.mont(m)), 1, H.ptr(tab[0]), H.ptr(buf)))
out["verify_projective"] = measure(lambda: lib.h_verify(H.ptr(H.pt_mont(pk, z1)), H.ptr(H.limbs(u)), H.ptr(H.pt_mont(Rp, z2)), H.ptr(H.mont(m)), 0, H.ptr(tab[0]), H.ptr(buf)))
uv = np.zeros(16, np.uint32); uo = np.zeros(8, np.uint32)
out["sign"] = measure(lambda: lib.h_sign(H.ptr(H.limbs(sk)), H.ptr(H.limbs(nonce)), H.ptr(H.mont(m)), H.ptr(tab[0]), H.ptr(uo), H.ptr(uv), H.ptr(buf)))
uvp = np.zeros(16, np.uint32)
out["sign_double"] = measure(lambda: lib.h_sign_double(H.ptr(H.limbs(sk)), H.ptr(H.limbs(nonce)), H.ptr(H.mont(m)), H.ptr(tab[0]), H.ptr(tab[1]), H.ptr(uo), H.ptr(uv), H.ptr(uvp), H.ptr(buf)))
ud, Rd, Rdp, cd = o.sign_double(sk, nonce, m, mul=V.mul)
pkp = V.mul(o.G_NUMS, sk)
out["verify_double_affine"] = measure(lambda: lib.h_verify_double(H.ptr(H.pt_mont(pk)), H.ptr(H.pt_mont(pkp)), H.ptr(H.limbs(ud)), H.ptr(H.pt_mont(Rd)), H.ptr(H.pt_mont(Rdp)), H.ptr(H.mont(m)), 1, H.ptr(tab[0]), H.ptr(tab[1]), H.ptr(buf)))
gen = V.mul(o.G, rnd.randrange(o.R)); pkv = V.mul(gen, sk)
uvg, Rvg, cvg = o.sign_vargen(sk, gen, nonce, m, mul=V.mul)
out["verify_vargen_affine"] = measure(lambda: lib.h_verify_vargen(H.ptr(H.pt_mont(pkv)), H.ptr(H.pt_mont(gen)), H.ptr(H.limbs(uvg)), H.ptr(H.pt_mont(Rvg)), H.ptr(H.mont(m)), 1, H.ptr(buf)))
# building blocks of the composite entries below
out["fq_inv"] = measure(lambda: lib.h_fq_inv(H.ptr(H.mont(12345)), H.ptr(buf)))  # Fermat: the address-oblivious paths and table builds
out["fq_inv_euclid"] = measure(lambda: lib.h_fq_inv_fast(H.ptr(H.mont(rnd.randrange(o.Q))), H.ptr(buf)))  # inv.cuh: what the kernels use (count varies a little with the input)
pkbytes = np.frombuffer(o.affine_to_bytes(pk), np.uint32).copy()
out["decompress"] = measure(lambda: lib.h_decompress(H.ptr(pkbytes), H.ptr(uv)))
# what k_fixed_batch<OP_SIGN> EXECUTES per signature: 4 signatures share one (Euclidean) inversion (Montgomery's trick:
# 3 (k - 1) extra products per k points), so 3/4 of an inversion disappears from the one-tuple body counted above
K = 4
sb = dict(out["sign"])
sb["imad_wide_per_tuple"] = out["sign"]["imad_wide_per_tuple"] - (K - 1) * out["fq_inv_euclid"]["imad_wide_per_tuple"] // K + 3 * (K - 1) * 120 // K
sb["fq_mul"] = out["sign"]["fq_mul"] - (K - 1) * out["fq_inv_euclid"]["fq_mul"] // K + 3 * (K - 1) // K
sb["fq_sqr"] = out["sign"]["fq_sqr"] - (K - 1) * out["fq_inv_euclid"]["fq_sqr"] // K
sb["note"] = "executed count of k_fixed_batch<OP_SIGN>: one shared inversion per 4 signatures (the one-tuple body is `sign`)"
out["sign_batch4"] = sb
# byte-level verify = two decompressions (decode kernel) + the limb-level verification; canonical -> Montgomery of the message: 1 product
vb = {k: out["verify_affine"][k] + 2 * out["decompress"][k] for k in ("imad_wide_per_tuple", "fq_mul", "fq_sqr", "fq_dot5", "fq_addsub", "fr_mont_mul", "dfma")}
vb["imad_wide_per_tuple"] += 120
vb["fq_mul"] += 1
vb["note"] = "decode kernel (2 point decompressions + message to Montgomery form) + challenge kernel + curve kernel"
out["verify_bytes"] = vb
# verifier-side witness rows (core.cuh verify_witness_core) of valid signatures, affine inputs: u G by comb (u G' too), u GEN
# and c PK by 64-window variable-base multiplication, two batched Euclidean inversions
rows = np.zeros(8 * 19, np.uint32)
nul = np.zeros(24, np.uint32)
out["verify_witness_single"] = measure(lambda: lib.h_verify_witness(0, H.ptr(H.pt_mont(pk)), H.ptr(nul), H.ptr(H.limbs(u)), H.ptr(H.pt_mont(Rp)), H.ptr(nul), H.ptr(H.mont(m)), 1, 0, H.ptr(tab[0]), H.ptr(tab[1]), H.ptr(rows)))
out["verify_witness_double"] = measure(lambda: lib.h_verify_witness(1, H.ptr(H.pt_mont(pk)), H.ptr(H.pt_mont(pkp)), H.ptr(H.limbs(ud)), H.ptr(H.pt_mont(Rd)), H.ptr(H.pt_mont(Rdp)), H.ptr(H.mont(m)), 1, 0, H.ptr(tab[0]), H.ptr(tab[1]), H.ptr(rows)))
out["verify_witness_vargen"] = measure(lambda: lib.h_verify_witness(2, H.ptr(H.pt_mont(pkv)), H.ptr(H.pt_mont(gen)), H.ptr(H.limbs(uvg)), H.ptr(H.pt_mont(Rvg)), H.ptr(nul), H.ptr(H.mont(m)), 1, 0, H.ptr(tab[0]), H.ptr(tab[1]), H.ptr(rows)))
# verification against a registered key (core.cuh verify_keyset_core, tests/host_keyset.cpp) of valid signatures, affine:
# the challenge hash, u G by the 16-bit comb (u G' too) or u GEN by the key's 8-bit comb, c PK by the key's 8-bit comb
sok = os.path.join(ROOT, "build", "host_keyset16.so")
subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-DSB_COMB_BITS=16", "-include",
                       os.path.join(ROOT, "tests", "host_shim.h"), "-o", sok, os.path.join(ROOT, "tests", "host_keyset.cpp")])
klib = ctypes.CDLL(sok)
H.setup_hades(klib)
klib.h_verify_keyset.argtypes = [ctypes.c_int, ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p, ctypes.c_uint32] + \
    [ctypes.c_void_p] * 4 + [ctypes.c_int, ctypes.c_int] + [ctypes.c_void_p] * 3
def ktabs(*pts):  # the keyset's combs of one key (the build is not counted)
    t = [np.zeros(32 * 129 * 24, np.uint32) for _ in pts]
    for x, p in zip(t, pts):
        klib.h_keyset_table(H.ptr(H.pt_mont(p)), 1, H.ptr(x))
    return np.concatenate(t)
kok = np.ones(1, np.uint32)
ks = [ktabs(pk), ktabs(pk, pkp), ktabs(pkv, gen)]
kargs = lambda s, uu, R1, R2: (s, H.ptr(ks[s]), 1, H.ptr(kok), 0, H.ptr(H.limbs(uu)), H.ptr(H.pt_mont(R1)), H.ptr(R2), H.ptr(H.mont(m)), 1, 0,
                               H.ptr(tab[0]), H.ptr(tab[1]), H.ptr(buf))
out["keyset_verify_single"] = measure(lambda: klib.h_verify_keyset(*kargs(0, u, Rp, nul)), klib)
out["keyset_verify_double"] = measure(lambda: klib.h_verify_keyset(*kargs(1, ud, Rd, H.pt_mont(Rdp))), klib)
out["keyset_verify_vargen"] = measure(lambda: klib.h_verify_keyset(*kargs(2, uvg, Rvg, nul)), klib)
st = np.concatenate([H.mont(x) for x in range(5)])
out["hades_perm_sparse"] = measure(lambda: lib.h_hades(H.ptr(st), 0))  # the production form: small-integer layers for the default MDS
out["hades_perm_dense"] = measure(lambda: lib.h_hades(H.ptr(st), 1))
out["_note"] = "counted by the instrumented host build of schnorr_b200/csrc (same per-tuple code as the kernels, 16-bit comb); 1 fq_mul = 120 IMAD.WIDE, 1 fq_sqr = 84, 1 fq_dot5 (5 products, 1 reduction) = 368, 1 fr_mont_mul = 128; dfma = FP64 fused multiply-adds of the small-integer Hades layers (hades.cuh, 1 per limb product of C s, plus the reductions); single-key verify also counts the 13 limb products of every step of the half-size-scalar Euclid (hgcd.cuh)"
if "--check" not in sys.argv:
    path = os.path.join(ROOT, "profiles", "op_counts.json")
    old = json.load(open(path)) if os.path.exists(path) else {}
    for k, v in out.items():
        if isinstance(v, dict) and isinstance(old.get(k), dict) and "dram_bytes_per_launch_ncu" in old[k]:
            v["dram_bytes_per_launch_ncu"] = old[k]["dram_bytes_per_launch_ncu"]
    json.dump(out, open(path, "w"), indent=1)
print(json.dumps(out, indent=1))
