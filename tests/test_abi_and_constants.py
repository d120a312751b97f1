"""The C-ABI library loads and exports every symbol include/schnorr_b200.h declares (no compute call here);
the generated constants header agrees with the oracle; host-side representation logic of the API mirror."""
import ctypes
import os
import random
import re

import numpy as np
import pytest

import schnorr_oracle as o

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
Q, R = o.Q, o.R


def _ensure_built():
    lib = os.path.join(ROOT, "schnorr_b200", "libschnorr_b200.so")
    if not os.path.exists(lib):
        import __graft_entry__ as g
        g.build()
    return lib


def test_library_exports_every_declared_symbol():
    path = _ensure_built()
    hdr = open(os.path.join(ROOT, "include", "schnorr_b200.h")).read()
    declared = sorted(set(re.findall(r"\b(sb200_[a-z0-9_]+)\s*\(", hdr)))
    assert len(declared) >= 22
    lib = ctypes.CDLL(path)
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in the header but not exported"
    from schnorr_b200 import _lib
    assert sorted(_lib.EXPORTED_SYMBOLS) == declared
    _lib.load_library()  # sets prototypes for all of them
    lib.sb200_strerror.restype = ctypes.c_char_p
    assert lib.sb200_strerror(0) == b"ok" and b"argument" in lib.sb200_strerror(-1)


def test_no_cpu_fallback_without_gpu():
    """Engine([0]) raises when no device is visible; a child process with CUDA_VISIBLE_DEVICES empty sees none, so this
    holds on a GPU machine too"""
    import subprocess
    import sys
    _ensure_built()
    code = ("from schnorr_b200 import Engine, SchnorrB200Error\n"
            "try:\n    Engine([0])\nexcept SchnorrB200Error as e:\n    print('raised:', e)\n")
    out = subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True, timeout=120,
                         env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert out.returncode == 0, out.stdout + out.stderr
    assert "raised:" in out.stdout, out.stdout + out.stderr


def test_product_never_imports_the_oracle():
    for dirpath, _, files in os.walk(os.path.join(ROOT, "schnorr_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cpp")):
                src = open(os.path.join(dirpath, f), errors="ignore").read()
                assert "schnorr_oracle" not in src and "ref_cpu" not in src and "oracle/" not in src, f


def _parse(name, text):
    """field elements of `#define NAME {...}` (one-line) or `#define NAME { \\ ... }` (multi-line)"""
    lines = text.splitlines()
    i = next(k for k, l in enumerate(lines) if l.startswith("#define " + name + " "))
    body = lines[i]
    if lines[i].rstrip().endswith("\\"):
        j = i + 1
        while lines[j].strip() != "}":
            body += lines[j]
            j += 1
    words = [int(w, 16) for w in re.findall(r"0x([0-9a-f]{8})u", body)]
    return [sum(w << (32 * k) for k, w in enumerate(words[p:p + 8])) for p in range(0, len(words), 8)]


def test_generated_constants_match_oracle():
    text = open(os.path.join(ROOT, "schnorr_b200", "csrc", "constants_gen.cuh")).read()
    mont = lambda x: x * o.MONT_R % Q
    one_line = lambda n: _parse(n, text)[0]
    assert one_line("SB200_FQ_MOD_INIT") == Q and one_line("SB200_FR_MOD_INIT") == R
    assert one_line("SB200_FQ_ONE_INIT") == o.MONT_R % Q and one_line("SB200_FQ_R2_INIT") == o.MONT_R ** 2 % Q
    assert one_line("SB200_FR_R2_INIT") == o.MONT_R ** 2 % R
    assert one_line("SB200_ED_D_INIT") == mont(o.D) and one_line("SB200_ED_2D_INIT") == mont(2 * o.D % Q)
    assert (one_line("SB200_G_U_INIT"), one_line("SB200_G_V_INIT")) == (mont(o.G[0]), mont(o.G[1]))
    assert (one_line("SB200_GP_U_INIT"), one_line("SB200_GP_V_INIT")) == (mont(o.G_NUMS[0]), mont(o.G_NUMS[1]))
    assert "SB200_HADES_RC_INIT" not in text and "SB200_HADES_MDS_INIT" not in text  # inputs of sb200_init_ex now (test_params.py)
    ninv = int(re.search(r"#define SB200_FR_NINV 0x([0-9a-f]+)u", text).group(1), 16)
    assert (ninv * R + 1) % (1 << 32) == 0


def test_api_host_side_formats():
    from schnorr_b200 import api
    rnd = random.Random(6)
    # StdRng mirrors the oracle's (and so rand 0.8's known answers)
    a, b = api.StdRng.seed_from_u64(2321), o.StdRng.seed_from_u64(2321)
    assert [a.random_scalar() for _ in range(3)] == [b.random_fr() for _ in range(3)]
    assert a.random_bls() == b.random_fq()
    assert a.random_scalars(5) == [b.random_fr() for _ in range(5)]
    seed = bytes([1, 0, 0, 0, 23, 0, 0, 0, 200, 1, 0, 0, 210, 30, 0, 0] + [0] * 16)
    assert int.from_bytes(api.StdRng(seed).fill_bytes(8), "little") == 10719222850664546238
    # compressed points / signatures round-trip exactly like JubJubAffine::{to,from}_bytes
    for _ in range(10):
        k = rnd.randrange(R)
        P = o.pt_mul_fast(o.G, k)
        z = rnd.randrange(1, Q)
        E = api.JubJubExtended(P[0] * z, P[1] * z, z)
        assert E.to_bytes() == o.affine_to_bytes(P)
        assert api.JubJubExtended.from_bytes(E.to_bytes()) == E  # projective equality
        sig = api.Signature(k, E)
        assert api.Signature.from_bytes(sig.to_bytes()) == sig and len(sig.to_bytes()) == 64
        sd = api.SignatureDouble(k, E, api.JubJubExtended(*o.G_NUMS))
        assert api.SignatureDouble.from_bytes(sd.to_bytes()) == sd and len(sd.to_bytes()) == 96
    with pytest.raises(api.InvalidData):
        api.SecretKey.from_bytes(R.to_bytes(32, "little"))
    with pytest.raises(api.InvalidData):
        api.PublicKey.from_bytes(Q.to_bytes(32, "little"))
    bad_v = next(v for v in range(2, 100) if o.affine_from_bytes(v.to_bytes(32, "little")) is None)
    with pytest.raises(api.InvalidData):
        api.PublicKey.from_bytes(bad_v.to_bytes(32, "little"))
