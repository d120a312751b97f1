"""Host-side mirror of dusk-schnorr's public API on top of the CUDA engine.

The reference is a Rust crate and this image has no Rust toolchain, so the reference-facing host layer
is written here in Python with the SAME names, argument meaning and error behaviour
(`rust/` holds the Rust sources a maintainer would compile; INTEGRATION.md):

    SecretKey::{random, sign, sign_double, with_variable_generator, to_bytes, from_bytes}
                                                /root/reference/src/keys/secret.rs:56-263
    SecretKeyVarGen::{new, random, sign, ...}   /root/reference/src/keys/secret.rs:307-451
    PublicKey::{from(&SecretKey), verify, from_raw_unchecked, to_bytes, from_bytes}
                                                /root/reference/src/keys/public.rs:59-145
    PublicKeyDouble / PublicKeyVarGen           /root/reference/src/keys/public.rs:189-433
    Signature / SignatureDouble / SignatureVarGen::{u, R, R_prime, to_bytes, from_bytes}
                                                /root/reference/src/signatures.rs:58-404

Every scalar multiplication, hash and comparison runs on the GPU through the C ABI (single calls are
batches of one); only representation work stays on the host, as in the reference: byte
(de)serialisation, canonical<->Montgomery conversion and the RNG state.  The batch signers hand the RNG's
position to the device, which draws the nonces the host would have drawn and returns the advanced position.  There is no CPU fallback for the
arithmetic: without the CUDA library / a B200 the first call raises.

New relative to the reference: the `*_batch` class methods (what north_star calls the batch entry
points): they take sequences and return arrays, and are what a high-throughput caller uses.
"""
from __future__ import annotations

import struct
from typing import List, Optional, Sequence, Tuple

import numpy as np

from ._lib import Engine

Q = 0x73EDA753299D7D483339D80809A1D80553BDA402FFFE5BFEFFFFFFFF00000001
R = 0x0E7DB4EA6533AFA906673B0101343B00A6682093CCC81082D0970E5ED6F72CB7
_RADIX = 1 << 256
_RINV = pow(_RADIX, -1, Q)
_D = (-10240 * pow(10241, -1, Q)) % Q

_engine: Optional[Engine] = None


def get_engine() -> Engine:
    """Process-wide default engine on device 0 (created on first use; raises without a GPU)."""
    global _engine
    if _engine is None:
        _engine = Engine([0])
    return _engine


def set_engine(e: Optional[Engine]) -> None:
    global _engine
    _engine = e


class InvalidData(ValueError):
    """dusk_bytes::Error::InvalidData: non-canonical scalar or bytes that are not a curve point."""


# ---- representation helpers (host-side formats only) ---------------------------------------------
def _limbs(x: int) -> np.ndarray:
    return np.frombuffer(int(x).to_bytes(32, "little"), dtype=np.uint32)


def _int(a) -> int:
    return int.from_bytes(np.ascontiguousarray(a, dtype=np.uint32).tobytes(), "little")


def _mont(x: int) -> np.ndarray:
    return _limbs(x % Q * _RADIX % Q)


def _unmont(a) -> int:
    return _int(a) * _RINV % Q


def _scalars(xs: Sequence[int]) -> np.ndarray:
    out = np.empty((len(xs), 8), np.uint32)
    for i, x in enumerate(xs):
        out[i] = _limbs(x)
    return out


def _fqs(xs: Sequence[int]) -> np.ndarray:
    out = np.empty((len(xs), 8), np.uint32)
    for i, x in enumerate(xs):
        out[i] = _mont(x)
    return out


class JubJubExtended:
    """A JubJub point as the projective triple (U : V : Z), Z != 0 (what `JubJubExtended` is up to its
    t1/t2 bookkeeping).  Equality is projective, as in the reference (/root/reference/tests/keys.rs:52-58)."""
    __slots__ = ("U", "V", "Z")

    def __init__(self, U: int, V: int, Z: int = 1):
        self.U, self.V, self.Z = U % Q, V % Q, Z % Q

    @classmethod
    def identity(cls):
        return cls(0, 1, 1)

    def __eq__(self, o):
        return isinstance(o, JubJubExtended) and (self.U * o.Z - o.U * self.Z) % Q == 0 and (self.V * o.Z - o.V * self.Z) % Q == 0

    def __hash__(self):
        return hash(self.affine())

    def affine(self) -> Tuple[int, int]:
        zi = pow(self.Z, -1, Q)
        return self.U * zi % Q, self.V * zi % Q

    def limbs(self) -> np.ndarray:
        return np.concatenate([_mont(self.U), _mont(self.V), _mont(self.Z)])

    def to_bytes(self) -> bytes:
        """JubJubAffine::to_bytes: v little-endian, bit 255 = lowest bit of u."""
        u, v = self.affine()
        b = bytearray(v.to_bytes(32, "little"))
        b[31] |= (u & 1) << 7
        return bytes(b)

    @classmethod
    def from_bytes(cls, b: bytes) -> "JubJubExtended":
        """JubJubAffine::from_bytes: decompress; no subgroup check (reference behaviour)."""
        if len(b) != 32:
            raise InvalidData("bad length")
        sign = b[31] >> 7
        v = int.from_bytes(b, "little") & ((1 << 255) - 1)
        if v >= Q:
            raise InvalidData("non-canonical v")
        v2 = v * v % Q
        den = (1 + _D * v2) % Q
        u2 = (v2 - 1) * pow(den, -1, Q) % Q if den else 0
        u = _fq_sqrt(u2)
        if u is None:
            raise InvalidData("not on the curve")
        if (u & 1) != sign:
            u = (-u) % Q
        return cls(u, v, 1)


def _fq_sqrt(a: int) -> Optional[int]:
    a %= Q
    if a == 0:
        return 0
    if pow(a, (Q - 1) // 2, Q) != 1:
        return None
    s, t = 32, (Q - 1) >> 32
    z = 7
    while pow(z, (Q - 1) // 2, Q) != Q - 1:
        z += 1
    m, c, tt, r = s, pow(z, t, Q), pow(a, t, Q), pow(a, (t + 1) // 2, Q)
    while tt != 1:
        i, x = 0, tt
        while x != 1:
            x, i = x * x % Q, i + 1
        b = pow(c, 1 << (m - i - 1), Q)
        m, c = i, b * b % Q
        tt, r = tt * c % Q, r * b % Q
    return r


def _points(ps: Sequence[JubJubExtended]) -> np.ndarray:
    out = np.empty((len(ps), 24), np.uint32)
    for i, p in enumerate(ps):
        out[i] = p.limbs()
    return out


def _points_out(a: np.ndarray) -> List[JubJubExtended]:
    return [JubJubExtended(_unmont(r[:8]), _unmont(r[8:16]), 1) for r in np.asarray(a).reshape(-1, 16)]


def _scalar_from_bytes(b: bytes) -> int:
    x = int.from_bytes(b, "little")
    if len(b) != 32 or x >= R:
        raise InvalidData("non-canonical scalar")
    return x


# ---- RNG: rand 0.8 StdRng (ChaCha12), the stream the reference's tests consume -----------------
class StdRng:
    """`rand::rngs::StdRng` as far as the signing path draws from it: 64-byte little-endian draws.
    `random_scalar` = JubJubScalar::random, `random_bls` = BlsScalar::random (both from_bytes_wide)."""

    def __init__(self, seed: bytes):
        assert len(seed) == 32
        self.key = np.frombuffer(seed, dtype="<u4").astype(np.uint32)
        self.block = 0
        self.buf = b""

    @classmethod
    def seed_from_u64(cls, state: int) -> "StdRng":
        out = b""
        for _ in range(8):
            state = (state * 6364136223846793005 + 11634580027462260723) & 0xFFFFFFFFFFFFFFFF
            xs = (((state >> 18) ^ state) >> 27) & 0xFFFFFFFF
            rot = state >> 59
            out += struct.pack("<I", ((xs >> rot) | (xs << ((32 - rot) & 31))) & 0xFFFFFFFF)
        return cls(out)

    def blocks(self, first: int, count: int) -> np.ndarray:
        """ChaCha12 blocks [first, first+count) as a [count, 16] uint32 array (vectorised; seekable)."""
        ctr = np.arange(first, first + count, dtype=np.uint64)
        st = np.empty((16, count), np.uint32)
        st[0:4] = np.array([0x61707865, 0x3320646E, 0x79622D32, 0x6B206574], np.uint32)[:, None]
        st[4:12] = self.key[:, None]
        st[12], st[13] = (ctr & 0xFFFFFFFF).astype(np.uint32), (ctr >> np.uint64(32)).astype(np.uint32)
        st[14] = st[15] = 0
        x = st.copy()

        def rotl(v, n):
            return (v << np.uint32(n)) | (v >> np.uint32(32 - n))

        def qr(a, b, c, d):
            x[a] += x[b]; x[d] = rotl(x[d] ^ x[a], 16)
            x[c] += x[d]; x[b] = rotl(x[b] ^ x[c], 12)
            x[a] += x[b]; x[d] = rotl(x[d] ^ x[a], 8)
            x[c] += x[d]; x[b] = rotl(x[b] ^ x[c], 7)

        with np.errstate(over="ignore"):
            for _ in range(6):
                qr(0, 4, 8, 12); qr(1, 5, 9, 13); qr(2, 6, 10, 14); qr(3, 7, 11, 15)
                qr(0, 5, 10, 15); qr(1, 6, 11, 12); qr(2, 7, 8, 13); qr(3, 4, 9, 14)
            x += st
        return np.ascontiguousarray(x.T)

    @property
    def word_pos(self) -> int:
        """index of the next unread 32-bit keystream word (rand_chacha's `get_word_pos`); None when a byte draw of a
        length that is not a multiple of 4 left the stream inside a word"""
        return None if len(self.buf) % 4 else 16 * self.block - len(self.buf) // 4

    def seek(self, word_pos: int) -> None:
        """continue the stream at keystream word `word_pos` (rand_chacha's `set_word_pos`)"""
        self.block, off = divmod(int(word_pos), 16)
        self.buf = b""
        if off:
            self.buf = self.blocks(self.block, 1).tobytes()[4 * off:]
            self.block += 1

    def fill_bytes(self, n: int) -> bytes:
        while len(self.buf) < n:
            self.buf += self.blocks(self.block, 4).tobytes()
            self.block += 4
        out, self.buf = self.buf[:n], self.buf[n:]
        return out

    def next_u64(self) -> int:
        return int.from_bytes(self.fill_bytes(8), "little")

    def random_scalar(self) -> int:
        return int.from_bytes(self.fill_bytes(64), "little") % R

    def random_bls(self) -> int:
        return int.from_bytes(self.fill_bytes(64), "little") % Q

    def random_scalars(self, n: int) -> List[int]:
        """n consecutive JubJubScalar::random draws (= the nonces of n consecutive `sign` calls)."""
        raw = self.fill_bytes(64 * n)
        return [int.from_bytes(raw[64 * i:64 * i + 64], "little") % R for i in range(n)]


# ---- the reference's types -------------------------------------------------------------------------
class Signature:
    """/root/reference/src/signatures.rs:58-123"""
    SIZE = 64

    def __init__(self, u: int, R_: JubJubExtended):
        self._u, self._R = u, R_

    def u(self) -> int:
        return self._u

    def R(self) -> JubJubExtended:
        return self._R

    def __eq__(self, o):
        return type(o) is type(self) and self._u == o._u and self._R == o._R

    def to_bytes(self) -> bytes:
        return self._u.to_bytes(32, "little") + self._R.to_bytes()

    @classmethod
    def from_bytes(cls, b: bytes):
        if len(b) != cls.SIZE:
            raise InvalidData("bad length")
        return cls(_scalar_from_bytes(b[:32]), JubJubExtended.from_bytes(b[32:]))


class SignatureVarGen(Signature):
    """/root/reference/src/signatures.rs:337-404"""


class SignatureDouble:
    """/root/reference/src/signatures.rs:180-270"""
    SIZE = 96

    def __init__(self, u: int, R_: JubJubExtended, R_prime: JubJubExtended):
        self._u, self._R, self._Rp = u, R_, R_prime

    def u(self) -> int:
        return self._u

    def R(self) -> JubJubExtended:
        return self._R

    def R_prime(self) -> JubJubExtended:
        return self._Rp

    def __eq__(self, o):
        return isinstance(o, SignatureDouble) and (self._u, self._R, self._Rp) == (o._u, o._R, o._Rp)

    def to_bytes(self) -> bytes:
        return self._u.to_bytes(32, "little") + self._R.to_bytes() + self._Rp.to_bytes()

    @classmethod
    def from_bytes(cls, b: bytes):
        if len(b) != cls.SIZE:
            raise InvalidData("bad length")
        return cls(_scalar_from_bytes(b[:32]), JubJubExtended.from_bytes(b[32:64]), JubJubExtended.from_bytes(b[64:]))


class SecretKey:
    """/root/reference/src/keys/secret.rs:56-263"""
    SIZE = 32

    def __init__(self, scalar: int):
        self._s = scalar % R

    @classmethod
    def random(cls, rng: StdRng) -> "SecretKey":
        return cls(rng.random_scalar())

    def as_scalar(self) -> int:
        return self._s

    def __eq__(self, o):
        return isinstance(o, SecretKey) and self._s == o._s

    def to_bytes(self) -> bytes:
        return self._s.to_bytes(32, "little")

    @classmethod
    def from_bytes(cls, b: bytes):
        return cls(_scalar_from_bytes(b))

    def sign(self, rng: StdRng, msg: int) -> Signature:
        return SecretKey.sign_batch([self], rng, [msg])[0]

    def sign_double(self, rng: StdRng, message: int) -> SignatureDouble:
        return SecretKey.sign_double_batch([self], rng, [message])[0]

    def with_variable_generator(self, generator: JubJubExtended) -> "SecretKeyVarGen":
        return SecretKeyVarGen(self._s, generator)

    # batch entry points: signature i consumes the rng's i-th JubJubScalar::random draw, in order.  On a word boundary
    # (always, unless a byte draw of odd length came before) the device draws the nonces from the rng's position.
    @staticmethod
    def sign_batch(sks: Sequence["SecretKey"], rng: StdRng, msgs: Sequence[int]) -> List[Signature]:
        sk, m = _scalars([k._s for k in sks]), _fqs(msgs)
        if rng.word_pos is not None:
            u, Rr, _, pos = get_engine().sign_stdrng(0, sk, m, rng.key, rng.word_pos)
            rng.seek(pos)
        else:
            u, Rr, _ = get_engine().sign(sk, m, _scalars(rng.random_scalars(len(sks))))
        return [Signature(_int(u[i]), p) for i, p in enumerate(_points_out(Rr))]

    @staticmethod
    def sign_double_batch(sks: Sequence["SecretKey"], rng: StdRng, msgs: Sequence[int]) -> List[SignatureDouble]:
        sk, m = _scalars([k._s for k in sks]), _fqs(msgs)
        if rng.word_pos is not None:
            u, Rr, Rp, _, pos = get_engine().sign_stdrng(1, sk, m, rng.key, rng.word_pos)
            rng.seek(pos)
        else:
            u, Rr, Rp, _ = get_engine().sign_double(sk, m, _scalars(rng.random_scalars(len(sks))))
        return [SignatureDouble(_int(u[i]), a, b) for i, (a, b) in enumerate(zip(_points_out(Rr), _points_out(Rp)))]


class SecretKeyVarGen:
    """/root/reference/src/keys/secret.rs:307-451"""
    SIZE = 64

    def __init__(self, sk: int, generator: JubJubExtended):
        self._s, self._g = sk % R, generator

    @classmethod
    def new(cls, sk: int, generator: JubJubExtended):
        return cls(sk, generator)

    @classmethod
    def random(cls, rng: StdRng) -> "SecretKeyVarGen":
        sk = rng.random_scalar()
        scalar = rng.random_scalar()
        gen = _points_out(get_engine().dbg_scalar_mul(0, _scalars([scalar])))[0]  # GENERATOR_EXTENDED * scalar
        return cls(sk, gen)

    def secret_key(self) -> int:
        return self._s

    def generator(self) -> JubJubExtended:
        return self._g

    def __eq__(self, o):
        return isinstance(o, SecretKeyVarGen) and self._s == o._s and self._g == o._g

    def to_bytes(self) -> bytes:
        return self._s.to_bytes(32, "little") + self._g.to_bytes()

    @classmethod
    def from_bytes(cls, b: bytes):
        if len(b) != cls.SIZE:
            raise InvalidData("bad length")
        return cls(_scalar_from_bytes(b[:32]), JubJubExtended.from_bytes(b[32:]))

    def sign(self, rng: StdRng, msg: int) -> SignatureVarGen:
        return SecretKeyVarGen.sign_batch([self], rng, [msg])[0]

    @staticmethod
    def sign_batch(sks: Sequence["SecretKeyVarGen"], rng: StdRng, msgs: Sequence[int]) -> List[SignatureVarGen]:
        sk, gen, m = _scalars([k._s for k in sks]), _points([k._g for k in sks]), _fqs(msgs)
        if rng.word_pos is not None:
            u, Rr, _, pos = get_engine().sign_stdrng(2, sk, m, rng.key, rng.word_pos, gen=gen, affine=False)
            rng.seek(pos)
        else:
            u, Rr, _ = get_engine().sign_vargen(sk, gen, m, _scalars(rng.random_scalars(len(sks))), affine=False)
        return [SignatureVarGen(_int(u[i]), p) for i, p in enumerate(_points_out(Rr))]


class PublicKey:
    """/root/reference/src/keys/public.rs:59-145"""
    SIZE = 32

    def __init__(self, point: JubJubExtended):
        self._p = point

    @classmethod
    def from_secret_key(cls, sk: SecretKey) -> "PublicKey":  # `PublicKey::from(&sk)`
        return cls.from_secret_keys([sk])[0]

    @staticmethod
    def from_secret_keys(sks: Sequence[SecretKey]) -> List["PublicKey"]:
        return [PublicKey(p) for p in _points_out(get_engine().keygen(_scalars([k._s for k in sks])))]

    @classmethod
    def from_raw_unchecked(cls, key: JubJubExtended) -> "PublicKey":
        return cls(key)

    def as_ref(self) -> JubJubExtended:
        return self._p

    def __eq__(self, o):
        return isinstance(o, PublicKey) and self._p == o._p

    def to_bytes(self) -> bytes:
        return self._p.to_bytes()

    @classmethod
    def from_bytes(cls, b: bytes):
        return cls(JubJubExtended.from_bytes(b))

    def verify(self, sig: Signature, message: int) -> bool:
        return bool(PublicKey.verify_batch([self], [sig], [message])[0])

    @staticmethod
    def verify_batch(pks: Sequence["PublicKey"], sigs: Sequence[Signature], msgs: Sequence[int]) -> np.ndarray:
        ok, _ = get_engine().verify(_points([k._p for k in pks]), _scalars([s._u for s in sigs]),
                                    _points([s._R for s in sigs]), _fqs(msgs), affine=False, want_c=False)
        return ok


class PublicKeyDouble:
    """/root/reference/src/keys/public.rs:189-299"""
    SIZE = 64

    def __init__(self, pk: JubJubExtended, pk_prime: JubJubExtended):
        self._p, self._pp = pk, pk_prime

    @classmethod
    def from_secret_key(cls, sk: SecretKey) -> "PublicKeyDouble":
        a, b = get_engine().keygen_double(_scalars([sk._s]))
        return cls(_points_out(a)[0], _points_out(b)[0])

    @classmethod
    def from_raw_unchecked(cls, pk: JubJubExtended, pk_prime: JubJubExtended):
        return cls(pk, pk_prime)

    def pk(self) -> JubJubExtended:
        return self._p

    def pk_prime(self) -> JubJubExtended:
        return self._pp

    def __eq__(self, o):
        return isinstance(o, PublicKeyDouble) and self._p == o._p and self._pp == o._pp

    def to_bytes(self) -> bytes:
        return self._p.to_bytes() + self._pp.to_bytes()

    @classmethod
    def from_bytes(cls, b: bytes):
        if len(b) != cls.SIZE:
            raise InvalidData("bad length")
        return cls(JubJubExtended.from_bytes(b[:32]), JubJubExtended.from_bytes(b[32:]))

    def verify(self, sig_double: SignatureDouble, message: int) -> bool:
        return bool(PublicKeyDouble.verify_batch([self], [sig_double], [message])[0])

    @staticmethod
    def verify_batch(pks: Sequence["PublicKeyDouble"], sigs: Sequence[SignatureDouble], msgs: Sequence[int]) -> np.ndarray:
        ok, _ = get_engine().verify_double(_points([k._p for k in pks]), _points([k._pp for k in pks]),
                                           _scalars([s._u for s in sigs]), _points([s._R for s in sigs]),
                                           _points([s._Rp for s in sigs]), _fqs(msgs), affine=False, want_c=False)
        return ok


class PublicKeyVarGen:
    """/root/reference/src/keys/public.rs:331-433"""
    SIZE = 64

    def __init__(self, pk: JubJubExtended, generator: JubJubExtended):
        self._p, self._g = pk, generator

    @classmethod
    def from_secret_key(cls, sk: SecretKeyVarGen) -> "PublicKeyVarGen":
        pk = get_engine().keygen_vargen(_scalars([sk._s]), _points([sk._g]), affine=False)
        return cls(_points_out(pk)[0], sk._g)

    @classmethod
    def from_raw_unchecked(cls, pk: JubJubExtended, generator: JubJubExtended):
        return cls(pk, generator)

    def public_key(self) -> JubJubExtended:
        return self._p

    def generator(self) -> JubJubExtended:
        return self._g

    def __eq__(self, o):
        return isinstance(o, PublicKeyVarGen) and self._p == o._p and self._g == o._g

    def to_bytes(self) -> bytes:
        return self._p.to_bytes() + self._g.to_bytes()

    @classmethod
    def from_bytes(cls, b: bytes):
        if len(b) != cls.SIZE:
            raise InvalidData("bad length")
        return cls(JubJubExtended.from_bytes(b[:32]), JubJubExtended.from_bytes(b[32:]))

    def verify(self, sig_var_gen: SignatureVarGen, message: int) -> bool:
        return bool(PublicKeyVarGen.verify_batch([self], [sig_var_gen], [message])[0])

    @staticmethod
    def verify_batch(pks: Sequence["PublicKeyVarGen"], sigs: Sequence[SignatureVarGen], msgs: Sequence[int]) -> np.ndarray:
        ok, _ = get_engine().verify_vargen(_points([k._p for k in pks]), _points([k._g for k in pks]),
                                           _scalars([s._u for s in sigs]), _points([s._R for s in sigs]), _fqs(msgs),
                                           affine=False, want_c=False)
        return ok


class PublicKeySet:
    """A fixed set of public keys of one type (PublicKey, PublicKeyDouble or PublicKeyVarGen) registered once on the
    device (include/schnorr_b200_keyset.h), for callers that verify many signatures of the same keys: each key gets
    fixed-base tables, so a verification no longer multiplies by the key as a fresh point.  Not in the reference: an
    addition of this library.  `verify_batch(indices, sigs, msgs)` returns what the type's
    `verify_batch([keys[i] for i in indices], sigs, msgs)` returns (a key not on the curve verifies nothing)."""

    _SCHEMES = {PublicKey: 0, PublicKeyDouble: 1, PublicKeyVarGen: 2}

    def __init__(self, keys: Sequence):
        keys = list(keys)
        types = {type(k) for k in keys}
        if len(types) != 1 or next(iter(types)) not in self._SCHEMES:
            raise TypeError("PublicKeySet: a non-empty sequence of PublicKey, PublicKeyDouble or PublicKeyVarGen, one type")
        self.keys = keys
        self.scheme = self._SCHEMES[types.pop()]
        pk2 = None
        if self.scheme == 1:
            pk2 = _points([k._pp for k in keys])
        elif self.scheme == 2:
            pk2 = _points([k._g for k in keys])
        self._ks = get_engine().keyset(self.scheme, _points([k._p for k in keys]), pk2, affine=False)

    def __len__(self):
        return len(self.keys)

    def close(self):
        self._ks.close()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def verify_batch(self, indices: Sequence[int], sigs: Sequence, msgs: Sequence[int]) -> np.ndarray:
        idx = np.asarray(indices, dtype=np.int64).reshape(-1)
        if idx.size and (idx.min() < 0 or idx.max() >= len(self.keys)):
            raise IndexError("PublicKeySet.verify_batch: key index out of range")
        Rp = _points([s._Rp for s in sigs]) if self.scheme == 1 else None
        ok, _ = self._ks.verify(idx.astype(np.uint32), _scalars([s._u for s in sigs]), _points([s._R for s in sigs]), _fqs(msgs),
                                Rp=Rp, affine=False, want_c=False)
        return ok
