"""ctypes binding of libschnorr_b200.so (the C ABI in include/schnorr_b200.h).

There is no CPU fallback: if the CUDA library is missing or no B200 is visible, construction of an
`Engine` raises.  numpy arrays are the host buffers (uint32, C-contiguous, 16-byte aligned).
"""
from __future__ import annotations

import ctypes
import os
import weakref
from typing import Optional, Sequence

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SB200_LIB", os.path.join(_HERE, "libschnorr_b200.so"))  # override: kernel-variant experiments

POINTS_PROJECTIVE = 0
POINTS_AFFINE = 1
DEVICE_PTRS = 2
VERIFY_DUAL_PIPE = 4  # sb200_verify, SB_EXPERIMENTAL_FD builds only: warp-specialised kernel (hash warps on the FP64 pipe)
CHECK_POINTS = 8      # verify*: on-curve / Z != 0 check of every input point on the device
SIGN_OBLIVIOUS = 16   # sign* / keygen*: no address or branch depends on the nonce / secret key (shared-memory combs, masked scans)
ARK_CUMSUM, ARK_PLAIN, ARK_ENV = 0, 1, -1  # rules for the DEFAULT Hades round constants (include/schnorr_b200.h)
ERR_ARG, ERR_CUDA, ERR_NODEV, ERR_NOMEM, ERR_PARAMS, ERR_BUSY = -1, -2, -3, -4, -5, -6


class Params(ctypes.Structure):
    """`sb200_params`: the two generators, the 335 Hades round constants and the MDS matrix, all as Montgomery limbs
    (= dusk_bls12_381::BlsScalar's internal words).  Inputs of context creation, not baked constants."""
    _fields_ = [("struct_size", ctypes.c_uint32), ("reserved", ctypes.c_uint32),
                ("generator", ctypes.c_uint32 * 16), ("generator_nums", ctypes.c_uint32 * 16),
                ("round_constants", (ctypes.c_uint32 * 8) * 335), ("mds", ((ctypes.c_uint32 * 8) * 5) * 5)]

    def view(self, field: str) -> np.ndarray:
        """writable uint32 view of one field ([..., 8] limbs)"""
        a = np.ctypeslib.as_array(getattr(self, field))
        return a.reshape(-1, 8)


def default_params(ark: int = ARK_ENV) -> Params:
    """sb200_default_params: recalled generators, recipe-derived round constants (rule `ark`), Cauchy MDS."""
    lib = load_library()
    p = Params()
    rc = lib.sb200_default_params(ark, ctypes.byref(p))
    if rc != 0:
        raise SchnorrB200Error(f"sb200_default_params: {lib.sb200_strerror(rc).decode()}")
    return p


class StdRngPos(ctypes.Structure):
    """`sb200_stdrng`: a rand 0.8 StdRng (ChaCha12, stream 0) as its 32-byte seed (8 little-endian words) and the index
    of the next unread 32-bit keystream word (16 x block + word within the block)."""
    _fields_ = [("key", ctypes.c_uint32 * 8), ("word_pos", ctypes.c_uint64)]

    @classmethod
    def of(cls, key, word_pos: int) -> "StdRngPos":
        k = np.asarray(key, dtype=np.uint32).reshape(8)
        return cls((ctypes.c_uint32 * 8)(*[int(x) for x in k]), int(word_pos))


def _split_tables(out: np.ndarray) -> dict:
    cut = np.cumsum([0, 335, 25, 5, 649, 25])
    return {k: out[cut[i]:cut[i + 1]].copy() for i, k in enumerate(("rc", "mds", "pre", "sparse", "post"))}


def params_check(p: Params):
    """sb200_params_check (host only): (return code, derived Hades tables or None)"""
    lib = load_library()
    out = aligned_empty((1039, 8))
    rc = lib.sb200_params_check(ctypes.byref(p), out.ctypes.data)
    return rc, (_split_tables(out) if rc == 0 else None)


def ark_rule(name: Optional[str]) -> int:
    return {None: ARK_ENV, "env": ARK_ENV, "cumsum": ARK_CUMSUM, "plain": ARK_PLAIN}[name]


vp, u32p, i64, u32, ci = ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64, ctypes.c_uint32, ctypes.c_int
_PROTOTYPES = {  # every symbol of include/schnorr_b200.h: (restype, argtypes)
    "sb200_init": (ci, [ctypes.POINTER(ci), ci, ctypes.POINTER(vp)]),
    "sb200_init_ex": (ci, [vp, ctypes.POINTER(ci), ci, ctypes.POINTER(vp)]),
    "sb200_default_params": (ci, [ci, vp]),
    "sb200_get_params": (ci, [vp, vp]),
    "sb200_params_check": (ci, [vp, u32p]),
    "sb200_points_check": (ci, [vp, i64, u32] + [u32p] * 2),
    "sb200_sign_witness": (ci, [vp, i64, u32, ci] + [u32p] * 5),
    "sb200_dbg_verify_ec": (ci, [vp, i64, u32] + [u32p] * 5),
    "sb200_dbg_hades_tables": (ci, [vp, u32p]),
    "sb200_destroy": (None, [vp]),
    "sb200_strerror": (ctypes.c_char_p, [ci]),
    "sb200_last_error": (ctypes.c_char_p, [vp]),
    "sb200_device_count": (ci, [vp]),
    "sb200_set_stream": (ci, [vp, vp]),
    "sb200_launch_count": (ctypes.c_uint64, [vp]),
    "sb200_host_alloc": (ci, [ctypes.c_size_t, ctypes.POINTER(vp)]),
    "sb200_host_free": (None, [vp]),
    "sb200_verify": (ci, [vp, i64, u32] + [u32p] * 6),
    "sb200_verify_double": (ci, [vp, i64, u32] + [u32p] * 8),
    "sb200_verify_vargen": (ci, [vp, i64, u32] + [u32p] * 7),
    "sb200_sign": (ci, [vp, i64, u32] + [u32p] * 6),
    "sb200_sign_double": (ci, [vp, i64, u32] + [u32p] * 7),
    "sb200_sign_vargen": (ci, [vp, i64, u32] + [u32p] * 7),
    "sb200_keygen": (ci, [vp, i64, u32] + [u32p] * 2),
    "sb200_keygen_double": (ci, [vp, i64, u32] + [u32p] * 3),
    "sb200_keygen_vargen": (ci, [vp, i64, u32] + [u32p] * 3),
    "sb200_points_decompress": (ci, [vp, i64, u32] + [u32p] * 3),
    "sb200_points_compress": (ci, [vp, i64, u32] + [u32p] * 2),
    "sb200_scalars_from_wide": (ci, [vp, i64, u32, ci] + [u32p] * 2),
    "sb200_stdrng_random": (ci, [vp, i64, u32, ci, vp, u32p]),
    "sb200_sign_stdrng": (ci, [vp, i64, u32, ci] + [u32p] * 3 + [vp] + [u32p] * 4),
    "sb200_fq_to_mont": (ci, [vp, i64, u32] + [u32p] * 2),
    "sb200_fq_from_mont": (ci, [vp, i64, u32] + [u32p] * 2),
    "sb200_verify_bytes": (ci, [vp, i64, u32] + [u32p] * 5),
    "sb200_sign_bytes": (ci, [vp, i64, u32] + [u32p] * 5),
    "sb200_verify_double_bytes": (ci, [vp, i64, u32] + [u32p] * 5),
    "sb200_verify_vargen_bytes": (ci, [vp, i64, u32] + [u32p] * 5),
    "sb200_sign_double_bytes": (ci, [vp, i64, u32] + [u32p] * 5),
    "sb200_sign_vargen_bytes": (ci, [vp, i64, u32] + [u32p] * 5),
    "sb200_dbg_fq": (ci, [vp, i64, ci] + [u32p] * 3),
    "sb200_dbg_fr_mul": (ci, [vp, i64] + [u32p] * 3),
    "sb200_dbg_lattice3": (ci, [vp, i64] + [u32p] * 3),
    "sb200_dbg_hades": (ci, [vp, i64, ci, u32p]),
    "sb200_dbg_scalar_mul": (ci, [vp, i64, u32, ci] + [u32p] * 3),
}
_WITNESS_PROTOTYPES = {  # every symbol of include/schnorr_b200_witness.h (verifier-side witness rows)
    "sb200_verify_witness": (ci, [vp, i64, u32, ci] + [u32p] * 8),
    "sb200_verify_witness_bytes": (ci, [vp, i64, u32, ci] + [u32p] * 6),
}
_KEYSET_PROTOTYPES = {  # every symbol of include/schnorr_b200_keyset.h (verification against registered keys)
    "sb200_keyset_create": (ci, [vp, ci, i64, u32, u32p, u32p, u32p, ctypes.POINTER(vp)]),
    "sb200_keyset_destroy": (None, [vp]),
    "sb200_verify_keyset": (ci, [vp, vp, i64, u32] + [u32p] * 7),
}
_KEYSET_LIVE_PROTOTYPES = {  # every symbol of include/schnorr_b200_keyset_live.h (byte-level keysets, live updates)
    "sb200_verify_keyset_bytes": (ci, [vp, vp, i64, u32] + [u32p] * 5),
    "sb200_keyset_create_bytes": (ci, [vp, ci, i64, u32, u32p, u32p, ctypes.POINTER(vp)]),
    "sb200_keyset_update": (ci, [vp, i64, u32] + [u32p] * 4),
    "sb200_keyset_update_bytes": (ci, [vp, i64, u32] + [u32p] * 3),
    "sb200_keyset_revoke": (ci, [vp, i64, u32p]),
}
_KEYSET_WITNESS_PROTOTYPES = {  # every symbol of include/schnorr_b200_keyset_witness.h (witness rows against a keyset)
    "sb200_verify_witness_keyset": (ci, [vp, vp, i64, u32] + [u32p] * 7),
    "sb200_verify_witness_keyset_bytes": (ci, [vp, vp, i64, u32] + [u32p] * 6),
}
del vp, u32p, i64, u32, ci
EXPORTED_SYMBOLS = list(_PROTOTYPES)  # the symbols of include/schnorr_b200.h

_lib = None


class SchnorrB200Error(RuntimeError):
    pass


def load_library() -> ctypes.CDLL:
    """Load the shared library (no CUDA call is made until an Engine is created)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise SchnorrB200Error(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a). There is no CPU fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in {**_PROTOTYPES, **_WITNESS_PROTOTYPES, **_KEYSET_PROTOTYPES, **_KEYSET_LIVE_PROTOTYPES,
                              **_KEYSET_WITNESS_PROTOTYPES}.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export a declared symbol
        fn.restype, fn.argtypes = res, args
    _lib = lib
    return lib


def aligned_empty(shape, dtype=np.uint32, align=64) -> np.ndarray:
    n = int(np.prod(shape)) * np.dtype(dtype).itemsize
    raw = np.empty(n + align, dtype=np.uint8)
    off = (-raw.ctypes.data) % align
    return raw[off:off + n].view(dtype).reshape(shape)


class PinnedBuffer:
    """page-locked host memory from sb200_host_alloc, exposed as a numpy array (`.array`); freed on close() / GC"""

    def __init__(self, shape, dtype=np.uint32):
        lib = load_library()
        self._lib = lib
        nbytes = max(int(np.prod(shape)) * np.dtype(dtype).itemsize, 1)
        p = ctypes.c_void_p()
        rc = lib.sb200_host_alloc(nbytes, ctypes.byref(p))
        if rc != 0:
            raise SchnorrB200Error(f"sb200_host_alloc: {lib.sb200_strerror(rc).decode()}")
        self._p = p
        buf = (ctypes.c_uint8 * nbytes).from_address(p.value)
        self.array = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)

    def close(self):
        if getattr(self, "_p", None):
            self.array = None
            self._lib.sb200_host_free(self._p)
            self._p = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _arr(a, words: Optional[int], n: int, name: str) -> np.ndarray:
    a = np.asarray(a)
    if a.dtype != np.uint32:
        raise SchnorrB200Error(f"{name}: expected uint32 limbs, got {a.dtype}")
    if words is not None and a.size != n * words:
        raise SchnorrB200Error(f"{name}: expected {n} x {words} u32, got {a.size}")
    if not a.flags["C_CONTIGUOUS"] or a.ctypes.data % 16:
        b = aligned_empty(a.shape)
        b[...] = a
        a = b
    return a


class Engine:
    """One sb200 context: comb tables for G and G' resident on each device, two streams per device."""

    def __init__(self, devices: Optional[Sequence[int]] = None, params: Optional[Params] = None, ark: Optional[str] = None):
        """`params`: an explicit sb200_params (e.g. the real crate's tables); else the defaults under round-constant
        rule `ark` ("cumsum" | "plain" | None = environment variable SB200_ARK, default cumsum)."""
        self._lib = load_library()
        devs = list(devices) if devices is not None else [0]
        arr = (ctypes.c_int * len(devs))(*devs)
        h = ctypes.c_void_p()
        self.params = params if params is not None else default_params(ark_rule(ark))
        rc = self._lib.sb200_init_ex(ctypes.byref(self.params), arr, len(devs), ctypes.byref(h))
        if rc != 0:
            err = SchnorrB200Error(f"sb200_init_ex failed: {self._lib.sb200_strerror(rc).decode()} (no CPU fallback)")
            err.code = rc
            raise err
        self._h = h
        self.devices = devs
        self._keysets = weakref.WeakSet()

    def close(self):
        if getattr(self, "_h", None):
            for ks in list(self._keysets):  # sb200_destroy frees them: their handles die with the context
                ks._h = None
            self._lib.sb200_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int, what: str):
        if rc != 0:
            raise SchnorrB200Error(
                f"{what}: {self._lib.sb200_strerror(rc).decode()} {self._lib.sb200_last_error(self._h).decode()}")

    @property
    def launch_count(self) -> int:
        return int(self._lib.sb200_launch_count(self._h))

    def set_stream(self, cuda_stream: int):
        self._check(self._lib.sb200_set_stream(self._h, ctypes.c_void_p(cuda_stream)), "set_stream")

    # ---- raw pointer calls (device pointers with DEVICE_PTRS, used by bench.py) -------------
    def call(self, name: str, n: int, flags: int, *ptrs: Optional[int]):
        fn = getattr(self._lib, "sb200_" + name)
        self._check(fn(self._h, n, flags, *[ctypes.c_void_p(p) if p else None for p in ptrs]), name)

    # ---- numpy front-ends -----------------------------------------------------------------------
    @staticmethod
    def _pw(affine: bool) -> int:
        return 16 if affine else 24

    @staticmethod
    def _unpack_bits(bitmap: np.ndarray, n: int) -> np.ndarray:
        return np.unpackbits(bitmap.view(np.uint8), bitorder="little")[:n].astype(bool)

    def verify(self, pk, u, R, msg, affine=True, want_c=True, dual_pipe=False, check_points=False):
        n = np.asarray(u).size // 8
        pw, fl = self._pw(affine), (POINTS_AFFINE if affine else POINTS_PROJECTIVE) | (VERIFY_DUAL_PIPE if dual_pipe else 0) | (CHECK_POINTS if check_points else 0)
        pk, u, R, msg = _arr(pk, pw, n, "pk"), _arr(u, 8, n, "u"), _arr(R, pw, n, "R"), _arr(msg, 8, n, "msg")
        bm = aligned_empty(((n + 31) // 32,)); bm[...] = 0
        c = aligned_empty((n, 8)) if want_c else None
        self.call("verify", n, fl, pk.ctypes.data, u.ctypes.data, R.ctypes.data, msg.ctypes.data, bm.ctypes.data,
                  c.ctypes.data if want_c else None)
        return self._unpack_bits(bm, n), c

    def verify_double(self, pk, pkp, u, R, Rp, msg, affine=True, want_c=True, check_points=False):
        n = np.asarray(u).size // 8
        pw, fl = self._pw(affine), (POINTS_AFFINE if affine else POINTS_PROJECTIVE) | (CHECK_POINTS if check_points else 0)
        pk, pkp, R, Rp = _arr(pk, pw, n, "pk"), _arr(pkp, pw, n, "pk'"), _arr(R, pw, n, "R"), _arr(Rp, pw, n, "R'")
        u, msg = _arr(u, 8, n, "u"), _arr(msg, 8, n, "msg")
        bm = aligned_empty(((n + 31) // 32,)); bm[...] = 0
        c = aligned_empty((n, 8)) if want_c else None
        self.call("verify_double", n, fl, pk.ctypes.data, pkp.ctypes.data, u.ctypes.data, R.ctypes.data, Rp.ctypes.data,
                  msg.ctypes.data, bm.ctypes.data, c.ctypes.data if want_c else None)
        return self._unpack_bits(bm, n), c

    def verify_vargen(self, pk, gen, u, R, msg, affine=True, want_c=True, check_points=False):
        n = np.asarray(u).size // 8
        pw, fl = self._pw(affine), (POINTS_AFFINE if affine else POINTS_PROJECTIVE) | (CHECK_POINTS if check_points else 0)
        pk, gen, R = _arr(pk, pw, n, "pk"), _arr(gen, pw, n, "gen"), _arr(R, pw, n, "R")
        u, msg = _arr(u, 8, n, "u"), _arr(msg, 8, n, "msg")
        bm = aligned_empty(((n + 31) // 32,)); bm[...] = 0
        c = aligned_empty((n, 8)) if want_c else None
        self.call("verify_vargen", n, fl, pk.ctypes.data, gen.ctypes.data, u.ctypes.data, R.ctypes.data, msg.ctypes.data,
                  bm.ctypes.data, c.ctypes.data if want_c else None)
        return self._unpack_bits(bm, n), c

    def sign(self, sk, msg, nonce, oblivious=False):
        n = np.asarray(sk).size // 8
        sk, msg, nonce = _arr(sk, 8, n, "sk"), _arr(msg, 8, n, "msg"), _arr(nonce, 8, n, "nonce")
        u, R, c = aligned_empty((n, 8)), aligned_empty((n, 16)), aligned_empty((n, 8))
        self.call("sign", n, SIGN_OBLIVIOUS if oblivious else 0, sk.ctypes.data, msg.ctypes.data, nonce.ctypes.data, u.ctypes.data, R.ctypes.data, c.ctypes.data)
        return u, R, c

    def sign_double(self, sk, msg, nonce, oblivious=False):
        n = np.asarray(sk).size // 8
        sk, msg, nonce = _arr(sk, 8, n, "sk"), _arr(msg, 8, n, "msg"), _arr(nonce, 8, n, "nonce")
        u, R, Rp, c = aligned_empty((n, 8)), aligned_empty((n, 16)), aligned_empty((n, 16)), aligned_empty((n, 8))
        self.call("sign_double", n, SIGN_OBLIVIOUS if oblivious else 0, sk.ctypes.data, msg.ctypes.data, nonce.ctypes.data, u.ctypes.data, R.ctypes.data,
                  Rp.ctypes.data, c.ctypes.data)
        return u, R, Rp, c

    def sign_vargen(self, sk, gen, msg, nonce, affine=True, oblivious=False):
        n = np.asarray(sk).size // 8
        pw, fl = self._pw(affine), (POINTS_AFFINE if affine else POINTS_PROJECTIVE) | (SIGN_OBLIVIOUS if oblivious else 0)
        sk, msg, nonce, gen = _arr(sk, 8, n, "sk"), _arr(msg, 8, n, "msg"), _arr(nonce, 8, n, "nonce"), _arr(gen, pw, n, "gen")
        u, R, c = aligned_empty((n, 8)), aligned_empty((n, 16)), aligned_empty((n, 8))
        self.call("sign_vargen", n, fl, sk.ctypes.data, gen.ctypes.data, msg.ctypes.data, nonce.ctypes.data, u.ctypes.data,
                  R.ctypes.data, c.ctypes.data)
        return u, R, c

    def keygen(self, sk, oblivious=False):
        n = np.asarray(sk).size // 8
        sk = _arr(sk, 8, n, "sk")
        pk = aligned_empty((n, 16))
        self.call("keygen", n, SIGN_OBLIVIOUS if oblivious else 0, sk.ctypes.data, pk.ctypes.data)
        return pk

    def keygen_double(self, sk, oblivious=False):
        n = np.asarray(sk).size // 8
        sk = _arr(sk, 8, n, "sk")
        pk, pkp = aligned_empty((n, 16)), aligned_empty((n, 16))
        self.call("keygen_double", n, SIGN_OBLIVIOUS if oblivious else 0, sk.ctypes.data, pk.ctypes.data, pkp.ctypes.data)
        return pk, pkp

    def keygen_vargen(self, sk, gen, affine=True, oblivious=False):
        n = np.asarray(sk).size // 8
        pw, fl = self._pw(affine), (POINTS_AFFINE if affine else POINTS_PROJECTIVE) | (SIGN_OBLIVIOUS if oblivious else 0)
        sk, gen = _arr(sk, 8, n, "sk"), _arr(gen, pw, n, "gen")
        pk = aligned_empty((n, 16))
        self.call("keygen_vargen", n, fl, sk.ctypes.data, gen.ctypes.data, pk.ctypes.data)
        return pk

    # ---- wire formats (bytes in / bytes out) ---------------------------------------------------------
    @staticmethod
    def _bytes_arr(b, width: int, name: str) -> np.ndarray:
        a = np.frombuffer(b, dtype=np.uint8) if isinstance(b, (bytes, bytearray, memoryview)) else np.asarray(b)
        a = a.view(np.uint8).reshape(-1, width)
        out = aligned_empty((a.shape[0], width), dtype=np.uint8)
        out[...] = a
        return out

    def points_decompress(self, data):
        """n x 32 bytes -> ([n,16] affine Montgomery limbs, ok[n])"""
        b = self._bytes_arr(data, 32, "bytes")
        n = b.shape[0]
        pts = aligned_empty((n, 16))
        bm = aligned_empty(((n + 31) // 32,)); bm[...] = 0
        self.call("points_decompress", n, 0, b.ctypes.data, pts.ctypes.data, bm.ctypes.data)
        return pts, self._unpack_bits(bm, n)

    def points_compress(self, points, affine=True):
        n = np.asarray(points).size // self._pw(affine)
        p = _arr(points, self._pw(affine), n, "points")
        out = aligned_empty((n, 32), dtype=np.uint8)
        self.call("points_compress", n, POINTS_AFFINE if affine else POINTS_PROJECTIVE, p.ctypes.data, out.ctypes.data)
        return out

    def scalars_from_wide(self, wide, field: int):
        """n x 64 bytes -> [n,8]: field 0 = JubJubScalar (canonical), 1 = BlsScalar (Montgomery)"""
        b = self._bytes_arr(wide, 64, "wide")
        n = b.shape[0]
        out = aligned_empty((n, 8))
        rc = self._lib.sb200_scalars_from_wide(self._h, n, 0, field, b.ctypes.data, out.ctypes.data)
        self._check(rc, "scalars_from_wide")
        return out

    def stdrng_random(self, key, word_pos: int, n: int, field: int, flags: int = 0, out=None):
        """n consecutive Field::random draws of the StdRng at (key, word_pos), computed on the device: [n, 8] limbs
        (field 0 = JubJubScalar canonical, 1 = BlsScalar Montgomery) and the advanced word position (word_pos + 16 n).
        With flags = DEVICE_PTRS, `out` is a device pointer and nothing is returned but the position."""
        pos = StdRngPos.of(key, word_pos)
        res = aligned_empty((n, 8)) if out is None else None
        rc = self._lib.sb200_stdrng_random(self._h, n, flags, field, ctypes.byref(pos), res.ctypes.data if res is not None else out)
        self._check(rc, "stdrng_random")
        return (res, pos.word_pos) if res is not None else pos.word_pos

    def sign_stdrng(self, scheme: int, sk, msg, key, word_pos: int, gen=None, affine=True, oblivious=False):
        """sign (scheme 0), sign_double (1) or sign_vargen (2) with nonce i = the i-th JubJubScalar::random draw of the
        StdRng at (key, word_pos), drawn on the device.  Returns the scheme's sign outputs (u, R[, R'], c) followed by
        the advanced word position."""
        n = np.asarray(sk).size // 8
        sk, msg = _arr(sk, 8, n, "sk"), _arr(msg, 8, n, "msg")
        fl = SIGN_OBLIVIOUS if oblivious else 0
        g = None
        if scheme == 2:
            fl |= POINTS_AFFINE if affine else POINTS_PROJECTIVE
            g = _arr(gen, self._pw(affine), n, "gen")
        u, R, c = aligned_empty((n, 8)), aligned_empty((n, 16)), aligned_empty((n, 8))
        Rp = aligned_empty((n, 16)) if scheme == 1 else None
        pos = StdRngPos.of(key, word_pos)
        rc = self._lib.sb200_sign_stdrng(self._h, n, fl, scheme, sk.ctypes.data, msg.ctypes.data,
                                         g.ctypes.data if g is not None else None, ctypes.byref(pos), u.ctypes.data,
                                         R.ctypes.data, Rp.ctypes.data if Rp is not None else None, c.ctypes.data)
        self._check(rc, "sign_stdrng")
        return ((u, R, Rp, c) if scheme == 1 else (u, R, c)) + (int(pos.word_pos),)

    def fq_to_mont(self, a):
        n = np.asarray(a).size // 8
        a = _arr(a, 8, n, "a")
        out = aligned_empty((n, 8))
        self.call("fq_to_mont", n, 0, a.ctypes.data, out.ctypes.data)
        return out

    def fq_from_mont(self, a):
        n = np.asarray(a).size // 8
        a = _arr(a, 8, n, "a")
        out = aligned_empty((n, 8))
        self.call("fq_from_mont", n, 0, a.ctypes.data, out.ctypes.data)
        return out

    def verify_bytes(self, pk, sig, msg):
        """pk n x 32, sig n x 64, msg n x 32 (canonical) -> (verdict[n], invalid[n])"""
        pk, sig, msg = self._bytes_arr(pk, 32, "pk"), self._bytes_arr(sig, 64, "sig"), self._bytes_arr(msg, 32, "msg")
        n = pk.shape[0]
        bm = aligned_empty(((n + 31) // 32,)); bm[...] = 0
        inv = aligned_empty(((n + 31) // 32,)); inv[...] = 0
        self.call("verify_bytes", n, 0, pk.ctypes.data, sig.ctypes.data, msg.ctypes.data, bm.ctypes.data, inv.ctypes.data)
        return self._unpack_bits(bm, n), self._unpack_bits(inv, n)

    def sign_bytes(self, sk, msg, nonce, want_invalid=False):
        """sk, msg, nonce n x 32 -> sig n x 64 [, invalid[n]: a from_bytes of the tuple fails; its signature is all zero]"""
        sk, msg, nonce = self._bytes_arr(sk, 32, "sk"), self._bytes_arr(msg, 32, "msg"), self._bytes_arr(nonce, 32, "nonce")
        n = sk.shape[0]
        out = aligned_empty((n, 64), dtype=np.uint8)
        inv = aligned_empty(((n + 31) // 32,)); inv[...] = 0
        self.call("sign_bytes", n, 0, sk.ctypes.data, msg.ctypes.data, nonce.ctypes.data, out.ctypes.data, inv.ctypes.data)
        return (out, self._unpack_bits(inv, n)) if want_invalid else out

    def _verify_bytes_generic(self, name, pk, pkw, sig, sigw, msg):
        pk, sig, msg = self._bytes_arr(pk, pkw, "pk"), self._bytes_arr(sig, sigw, "sig"), self._bytes_arr(msg, 32, "msg")
        n = pk.shape[0]
        bm = aligned_empty(((n + 31) // 32,)); bm[...] = 0
        inv = aligned_empty(((n + 31) // 32,)); inv[...] = 0
        self.call(name, n, 0, pk.ctypes.data, sig.ctypes.data, msg.ctypes.data, bm.ctypes.data, inv.ctypes.data)
        return self._unpack_bits(bm, n), self._unpack_bits(inv, n)

    def verify_double_bytes(self, pk, sig, msg):
        """pk n x 64 (pk || pk'), sig n x 96 (u || R || R'), msg n x 32 -> (verdict[n], invalid[n])"""
        return self._verify_bytes_generic("verify_double_bytes", pk, 64, sig, 96, msg)

    def verify_vargen_bytes(self, pk, sig, msg):
        """pk n x 64 (pk || generator), sig n x 64 (u || R), msg n x 32 -> (verdict[n], invalid[n])"""
        return self._verify_bytes_generic("verify_vargen_bytes", pk, 64, sig, 64, msg)

    def sign_double_bytes(self, sk, msg, nonce, want_invalid=False):
        sk, msg, nonce = self._bytes_arr(sk, 32, "sk"), self._bytes_arr(msg, 32, "msg"), self._bytes_arr(nonce, 32, "nonce")
        n = sk.shape[0]
        out = aligned_empty((n, 96), dtype=np.uint8)
        inv = aligned_empty(((n + 31) // 32,)); inv[...] = 0
        self.call("sign_double_bytes", n, 0, sk.ctypes.data, msg.ctypes.data, nonce.ctypes.data, out.ctypes.data, inv.ctypes.data)
        return (out, self._unpack_bits(inv, n)) if want_invalid else out

    def sign_vargen_bytes(self, sk, msg, nonce):
        """sk n x 64 (sk || generator) -> (sig n x 64, ok[n]: every from_bytes of the tuple succeeds)"""
        sk, msg, nonce = self._bytes_arr(sk, 64, "sk"), self._bytes_arr(msg, 32, "msg"), self._bytes_arr(nonce, 32, "nonce")
        n = sk.shape[0]
        out = aligned_empty((n, 64), dtype=np.uint8)
        bm = aligned_empty(((n + 31) // 32,)); bm[...] = 0
        self.call("sign_vargen_bytes", n, 0, sk.ctypes.data, msg.ctypes.data, nonce.ctypes.data, out.ctypes.data, bm.ctypes.data)
        return out, ~self._unpack_bits(bm, n)

    WITNESS_WIDTH = (11, 19, 13)

    def sign_witness(self, scheme: int, sk, msg, nonce, gen=None, affine=True):
        """PLONK witness rows of n signatures ([n, W, 8] Montgomery limbs; W = 11 / 19 / 13 for scheme 0 single,
        1 double, 2 vargen): u, R(, R'), PK(, PK' | GEN), m, c, SA = u G, SB = c PK(, SA', SB')"""
        n = np.asarray(sk).size // 8
        sk, msg, nonce = _arr(sk, 8, n, "sk"), _arr(msg, 8, n, "msg"), _arr(nonce, 8, n, "nonce")
        fl = (POINTS_AFFINE if affine else POINTS_PROJECTIVE) if scheme == 2 else 0
        g = _arr(gen, self._pw(affine), n, "gen") if scheme == 2 else None
        w = self.WITNESS_WIDTH[scheme]
        out = aligned_empty((n, w, 8))
        rc = self._lib.sb200_sign_witness(self._h, n, fl, scheme, sk.ctypes.data, msg.ctypes.data, nonce.ctypes.data,
                                          g.ctypes.data if g is not None else None, out.ctypes.data)
        self._check(rc, "sign_witness")
        return out

    def verify_witness(self, scheme: int, pk, u, R, msg, pk2=None, Rp=None, affine=True, check_points=False):
        """witness rows of received signatures (include/schnorr_b200_witness.h): (ok[n], rows[n, W, 8]) with the row
        layout of sign_witness.  pk2 = PK' (scheme 1) or the generator (scheme 2); Rp = R' (scheme 1)."""
        n = np.asarray(u).size // 8
        pw = self._pw(affine)
        fl = (POINTS_AFFINE if affine else POINTS_PROJECTIVE) | (CHECK_POINTS if check_points else 0)
        pk, u, R, msg = _arr(pk, pw, n, "pk"), _arr(u, 8, n, "u"), _arr(R, pw, n, "R"), _arr(msg, 8, n, "msg")
        pk2 = _arr(pk2, pw, n, "pk2") if scheme in (1, 2) else None
        Rp = _arr(Rp, pw, n, "R'") if scheme == 1 else None
        bm = aligned_empty(((n + 31) // 32,)); bm[...] = 0
        rows = aligned_empty((n, self.WITNESS_WIDTH[scheme], 8))
        rc = self._lib.sb200_verify_witness(self._h, n, fl, scheme, pk.ctypes.data, pk2.ctypes.data if pk2 is not None else None,
                                            u.ctypes.data, R.ctypes.data, Rp.ctypes.data if Rp is not None else None,
                                            msg.ctypes.data, bm.ctypes.data, rows.ctypes.data)
        self._check(rc, "verify_witness")
        return self._unpack_bits(bm, n), rows

    def verify_witness_bytes(self, scheme: int, pk, sig, msg):
        """the byte-level inputs of verify_bytes / verify_double_bytes / verify_vargen_bytes -> (ok[n], invalid[n],
        rows[n, W, 8]); a tuple that does not decode has invalid set, verdict 0 and an all-zero row"""
        pk = self._bytes_arr(pk, (32, 64, 64)[scheme], "pk")
        sig, msg = self._bytes_arr(sig, (64, 96, 64)[scheme], "sig"), self._bytes_arr(msg, 32, "msg")
        n = pk.shape[0]
        bm = aligned_empty(((n + 31) // 32,)); bm[...] = 0
        inv = aligned_empty(((n + 31) // 32,)); inv[...] = 0
        rows = aligned_empty((n, self.WITNESS_WIDTH[scheme], 8))
        rc = self._lib.sb200_verify_witness_bytes(self._h, n, 0, scheme, pk.ctypes.data, sig.ctypes.data, msg.ctypes.data,
                                                  bm.ctypes.data, rows.ctypes.data, inv.ctypes.data)
        self._check(rc, "verify_witness_bytes")
        return self._unpack_bits(bm, n), self._unpack_bits(inv, n), rows

    def keyset(self, scheme: int, pk, pk2=None, affine=True) -> "KeySet":
        """register n_keys public keys (include/schnorr_b200_keyset.h): per-key comb tables built on every device.
        pk2 = PK' (scheme 1) or the keys' generators (scheme 2)."""
        return KeySet(self, scheme, pk, pk2, affine)

    def keyset_from_bytes(self, scheme: int, pk_bytes) -> "KeySet":
        """register n_keys public keys given as their to_bytes() form (include/schnorr_b200_keyset_live.h): 32 B per key
        for scheme 0, 64 B (pk || pk' or pk || generator) for schemes 1 and 2.  key_ok[k] = the key's from_bytes succeeds."""
        return KeySet(self, scheme, None, pk_bytes=pk_bytes)

    def points_check(self, points, affine=True):
        """ok[n]: point i is on the curve with Z != 0 (what CHECK_POINTS applies inside the verify calls)"""
        n = np.asarray(points).size // self._pw(affine)
        p = _arr(points, self._pw(affine), n, "points")
        bm = aligned_empty(((n + 31) // 32,)); bm[...] = 0
        self.call("points_check", n, POINTS_AFFINE if affine else POINTS_PROJECTIVE, p.ctypes.data, bm.ctypes.data)
        return self._unpack_bits(bm, n)

    # ---- building-block probes --------------------------------------------------------------------
    def dbg_verify_ec(self, pk, u, R, c, affine=True):
        """curve half of verify with caller-supplied challenges: verdict[i] = (u G + c PK == R)"""
        n = np.asarray(u).size // 8
        pw, fl = self._pw(affine), POINTS_AFFINE if affine else POINTS_PROJECTIVE
        pk, u, R, c = _arr(pk, pw, n, "pk"), _arr(u, 8, n, "u"), _arr(R, pw, n, "R"), _arr(c, 8, n, "c")
        bm = aligned_empty(((n + 31) // 32,)); bm[...] = 0
        self.call("dbg_verify_ec", n, fl, pk.ctypes.data, u.ctypes.data, R.ctypes.data, c.ctypes.data, bm.ctypes.data)
        return self._unpack_bits(bm, n)

    def dbg_hades_tables(self):
        """the Hades tables derived from this context's parameters: dict of [k, 8] Montgomery limb arrays"""
        out = aligned_empty((1039, 8))
        self._check(self._lib.sb200_dbg_hades_tables(self._h, out.ctypes.data), "dbg_hades_tables")
        return _split_tables(out)

    def dbg_fq(self, op: int, a, b=None):
        n = np.asarray(a).size // 8
        a = _arr(a, 8, n, "a")
        b = _arr(b, 8, n, "b") if b is not None else None
        out = aligned_empty((n, 8))
        rc = self._lib.sb200_dbg_fq(self._h, n, op, a.ctypes.data, b.ctypes.data if b is not None else None, out.ctypes.data)
        self._check(rc, "dbg_fq")
        return out

    def dbg_fr_mul(self, a, b):
        n = np.asarray(a).size // 8
        a, b = _arr(a, 8, n, "a"), _arr(b, 8, n, "b")
        out = aligned_empty((n, 8))
        self._check(self._lib.sb200_dbg_fr_mul(self._h, n, a.ctypes.data, b.ctypes.data, out.ctypes.data), "dbg_fr_mul")
        return out

    def dbg_lattice3(self, c, u):
        """(a, b, d, flags) rows of csrc/lat3.cuh run on the device: (n, 32) uint32"""
        n = np.asarray(c).size // 8
        c, u = _arr(c, 8, n, "c"), _arr(u, 8, n, "u")
        out = aligned_empty((n, 32))
        self._check(self._lib.sb200_dbg_lattice3(self._h, n, c.ctypes.data, u.ctypes.data, out.ctypes.data), "dbg_lattice3")
        return out

    def dbg_hades(self, states, dense=False):
        n = np.asarray(states).size // 40
        s = aligned_empty((n, 40)); s[...] = np.asarray(states, dtype=np.uint32).reshape(n, 40)
        self._check(self._lib.sb200_dbg_hades(self._h, n, int(dense), s.ctypes.data), "dbg_hades")
        return s

    def dbg_scalar_mul(self, base: int, k, points=None, affine=True):
        n = np.asarray(k).size // 8
        pw, fl = self._pw(affine), POINTS_AFFINE if affine else POINTS_PROJECTIVE
        k = _arr(k, 8, n, "k")
        p = _arr(points, pw, n, "points") if points is not None else None
        out = aligned_empty((n, 16))
        rc = self._lib.sb200_dbg_scalar_mul(self._h, n, fl, base, p.ctypes.data if p is not None else None, k.ctypes.data, out.ctypes.data)
        self._check(rc, "dbg_scalar_mul")
        return out


class KeySet:
    """Public keys registered on every device of an Engine (include/schnorr_b200_keyset.h): `key_ok` (bool[n_keys]: every
    point of the key is on the curve with Z != 0, kept current by update and revoke), `verify`, the calls of
    include/schnorr_b200_keyset_live.h: `verify_bytes`, `update`, `update_bytes`, `revoke`, and those of
    include/schnorr_b200_keyset_witness.h: `verify_witness`, `verify_witness_bytes`.  Frees its device memory on
    close() / exit / GC."""

    KEY_BYTES = (32, 64, 64)  # to_bytes() of PublicKey, PublicKeyDouble, PublicKeyVarGen
    SIG_BYTES = (64, 96, 64)  # to_bytes() of Signature, SignatureDouble, SignatureVarGen

    def __init__(self, engine: Engine, scheme: int, pk, pk2=None, affine=True, pk_bytes=None):
        h = ctypes.c_void_p()
        if pk_bytes is not None:
            b = engine._bytes_arr(pk_bytes, self.KEY_BYTES[scheme], "pk_bytes")
            n = b.shape[0]
            ok = aligned_empty(((n + 31) // 32 + 1,)); ok[...] = 0
            rc = engine._lib.sb200_keyset_create_bytes(engine._h, scheme, n, 0, b.ctypes.data, ok.ctypes.data, ctypes.byref(h))
        else:
            pw = engine._pw(affine)
            n = np.asarray(pk).size // pw
            pk = _arr(pk, pw, n, "pk")
            pk2 = _arr(pk2, pw, n, "pk2") if scheme in (1, 2) else None
            ok = aligned_empty(((n + 31) // 32 + 1,)); ok[...] = 0
            rc = engine._lib.sb200_keyset_create(engine._h, scheme, n, POINTS_AFFINE if affine else POINTS_PROJECTIVE, pk.ctypes.data,
                                                 pk2.ctypes.data if pk2 is not None else None, ok.ctypes.data, ctypes.byref(h))
        engine._check(rc, "keyset_create")
        self._engine, self._h, self.scheme, self.n_keys = engine, h, scheme, n
        self.key_ok = engine._unpack_bits(ok, n)
        engine._keysets.add(self)

    def close(self):
        if getattr(self, "_h", None):
            self._engine._lib.sb200_keyset_destroy(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def verify(self, key_index, u, R, msg, Rp=None, affine=True, want_c=True, check_points=False):
        """verdict i = the scheme's verify of (key key_index[i], u[i], R[i] (, Rp[i]), msg[i]): (ok[n], c[n, 8] or None).
        An index >= n_keys or a key that is not key_ok gives verdict 0."""
        e = self._engine
        if not self._h:
            raise SchnorrB200Error("verify: the keyset is closed")
        idx = _arr(np.asarray(key_index).astype(np.uint32).reshape(-1), None, 0, "key_index")
        n = idx.size
        pw = e._pw(affine)
        fl = (POINTS_AFFINE if affine else POINTS_PROJECTIVE) | (CHECK_POINTS if check_points else 0)
        u, R, msg = _arr(u, 8, n, "u"), _arr(R, pw, n, "R"), _arr(msg, 8, n, "msg")
        Rp = _arr(Rp, pw, n, "R'") if self.scheme == 1 else None
        bm = aligned_empty(((n + 31) // 32,)); bm[...] = 0
        c = aligned_empty((n, 8)) if want_c else None
        rc = e._lib.sb200_verify_keyset(e._h, self._h, n, fl, idx.ctypes.data, u.ctypes.data, R.ctypes.data,
                                        Rp.ctypes.data if Rp is not None else None, msg.ctypes.data, bm.ctypes.data,
                                        c.ctypes.data if want_c else None)
        e._check(rc, "verify_keyset")
        return e._unpack_bits(bm, n), c

    def _open(self, what: str) -> Engine:
        if not self._h:
            raise SchnorrB200Error(f"{what}: the keyset is closed")
        return self._engine

    @staticmethod
    def _slots(slots) -> np.ndarray:
        return _arr(np.asarray(slots).astype(np.uint32).reshape(-1), None, 0, "slots")

    def verify_bytes(self, key_index, sig_bytes, msg_bytes):
        """wire-format signatures (the type's to_bytes()) and 32-byte canonical messages against the keys key_index[i]:
        (ok[n], invalid[n]).  invalid = the signature's or the message's from_bytes fails; an index >= n_keys, a key that is
        not key_ok or a revoked slot gives verdict 0 with invalid 0."""
        e = self._open("verify_bytes")
        idx = self._slots(key_index)
        n = idx.size
        sig, msg = e._bytes_arr(sig_bytes, self.SIG_BYTES[self.scheme], "sig"), e._bytes_arr(msg_bytes, 32, "msg")
        if sig.shape[0] != n or msg.shape[0] != n:
            raise SchnorrB200Error(f"verify_bytes: {n} key indices, {sig.shape[0]} signatures, {msg.shape[0]} messages")
        bm = aligned_empty(((n + 31) // 32,)); bm[...] = 0
        inv = aligned_empty(((n + 31) // 32,)); inv[...] = 0
        rc = e._lib.sb200_verify_keyset_bytes(e._h, self._h, n, 0, idx.ctypes.data, sig.ctypes.data, msg.ctypes.data,
                                              bm.ctypes.data, inv.ctypes.data)
        e._check(rc, "verify_keyset_bytes")
        return e._unpack_bits(bm, n), e._unpack_bits(inv, n)

    def verify_witness(self, key_index, u, R, msg, Rp=None, affine=True, check_points=False):
        """witness rows of received signatures against the keys key_index[i] (include/schnorr_b200_keyset_witness.h):
        (ok[n], rows[n, W, 8]) with the layout and values of Engine.verify_witness on the gathered keys.  An index >=
        n_keys, a key that is not key_ok or u >= r gives an all-zero row and verdict 0."""
        e = self._open("verify_witness")
        idx = self._slots(key_index)
        n = idx.size
        pw = e._pw(affine)
        fl = (POINTS_AFFINE if affine else POINTS_PROJECTIVE) | (CHECK_POINTS if check_points else 0)
        u, R, msg = _arr(u, 8, n, "u"), _arr(R, pw, n, "R"), _arr(msg, 8, n, "msg")
        Rp = _arr(Rp, pw, n, "R'") if self.scheme == 1 else None
        bm = aligned_empty(((n + 31) // 32,)); bm[...] = 0
        rows = aligned_empty((n, Engine.WITNESS_WIDTH[self.scheme], 8))
        rc = e._lib.sb200_verify_witness_keyset(e._h, self._h, n, fl, idx.ctypes.data, u.ctypes.data, R.ctypes.data,
                                                Rp.ctypes.data if Rp is not None else None, msg.ctypes.data, bm.ctypes.data,
                                                rows.ctypes.data)
        e._check(rc, "verify_witness_keyset")
        return e._unpack_bits(bm, n), rows

    def verify_witness_bytes(self, key_index, sig_bytes, msg_bytes):
        """verify_witness on wire-format signatures and 32-byte canonical messages: (ok[n], invalid[n], rows[n, W, 8]);
        a tuple whose signature or message does not decode has invalid set, verdict 0 and an all-zero row"""
        e = self._open("verify_witness_bytes")
        idx = self._slots(key_index)
        n = idx.size
        sig, msg = e._bytes_arr(sig_bytes, self.SIG_BYTES[self.scheme], "sig"), e._bytes_arr(msg_bytes, 32, "msg")
        if sig.shape[0] != n or msg.shape[0] != n:
            raise SchnorrB200Error(f"verify_witness_bytes: {n} key indices, {sig.shape[0]} signatures, {msg.shape[0]} messages")
        bm = aligned_empty(((n + 31) // 32,)); bm[...] = 0
        inv = aligned_empty(((n + 31) // 32,)); inv[...] = 0
        rows = aligned_empty((n, Engine.WITNESS_WIDTH[self.scheme], 8))
        rc = e._lib.sb200_verify_witness_keyset_bytes(e._h, self._h, n, 0, idx.ctypes.data, sig.ctypes.data, msg.ctypes.data,
                                                      bm.ctypes.data, rows.ctypes.data, inv.ctypes.data)
        e._check(rc, "verify_witness_keyset_bytes")
        return e._unpack_bits(bm, n), e._unpack_bits(inv, n), rows

    def _updated(self, rc: int, what: str, slots: np.ndarray, ok: np.ndarray) -> np.ndarray:
        self._engine._check(rc, what)
        new = self._engine._unpack_bits(ok, slots.size)
        self.key_ok[slots] = new
        return new

    def update(self, slots, pk, pk2=None, affine=True) -> np.ndarray:
        """rebuild the distinct slots `slots` in place with m new keys (layout of the constructor): the new key_ok[m]"""
        e = self._open("update")
        s = self._slots(slots)
        m, pw = s.size, e._pw(affine)
        pk = _arr(pk, pw, m, "pk")
        pk2 = _arr(pk2, pw, m, "pk2") if self.scheme in (1, 2) else None
        ok = aligned_empty(((m + 31) // 32 + 1,)); ok[...] = 0
        rc = e._lib.sb200_keyset_update(self._h, m, POINTS_AFFINE if affine else POINTS_PROJECTIVE, s.ctypes.data, pk.ctypes.data,
                                        pk2.ctypes.data if pk2 is not None else None, ok.ctypes.data)
        return self._updated(rc, "keyset_update", s, ok)

    def update_bytes(self, slots, pk_bytes) -> np.ndarray:
        """update from the keys' to_bytes() form: the new key_ok[m] (False where a key does not decode)"""
        e = self._open("update_bytes")
        s = self._slots(slots)
        b = e._bytes_arr(pk_bytes, self.KEY_BYTES[self.scheme], "pk_bytes")
        if b.shape[0] != s.size:
            raise SchnorrB200Error(f"update_bytes: {s.size} slots, {b.shape[0]} keys")
        ok = aligned_empty(((s.size + 31) // 32 + 1,)); ok[...] = 0
        rc = e._lib.sb200_keyset_update_bytes(self._h, s.size, 0, s.ctypes.data, b.ctypes.data, ok.ctypes.data)
        return self._updated(rc, "keyset_update_bytes", s, ok)

    def revoke(self, slots) -> None:
        """clear the key_ok bits of the distinct slots `slots`: tuples naming them verify to False until an update"""
        e = self._open("revoke")
        s = self._slots(slots)
        e._check(e._lib.sb200_keyset_revoke(self._h, s.size, s.ctypes.data), "keyset_revoke")
        self.key_ok[s] = False
