"""What every compute entry point of the C ABI accepts, rejects and launches, pinned literally.

For each `sb200_*` compute call a valid small call is varied one argument at a time: each flag bit alone (the five
defined bits and one unknown bit), each pointer null, each array pointer 4 bytes off a 16-byte boundary, n = 0 and
n = -1.  The return codes are the table below, written out rather than derived from the library, so that a change to
the dispatch code cannot move them quietly.  A rejected call must leave its outputs and the StdRng position untouched,
launch nothing, and leave the context able to repeat the valid call bit for bit.

The kernel launches of every call (sb200_launch_count, which bench.py reports) are pinned per pipeline chunk, for host
buffers in one chunk and in several chunks, and for device pointers.
"""
import ctypes

import numpy as np
import pytest

import vectors as V
from test_gpu_scale_parity import CHUNK_MIN, host_chunks

pytestmark = pytest.mark.gpu

OK, ARG = 0, -1
FLAG_BITS = (1, 2, 4, 8, 16, 64)  # POINTS_AFFINE, DEVICE_PTRS, VERIFY_DUAL_PIPE, CHECK_POINTS, SIGN_OBLIVIOUS, unknown
N_SMALL = 70                      # one chunk, ragged warp
N_CHUNKS = 3 * CHUNK_MIN + 77     # several chunks, the last ragged

# Entry points: (id, C name without sb200_, takes flags, integer arguments after the flags, pointer arguments).
# A pointer argument is ("in", base array) | ("out", words per tuple) | ("bm",) a bitmap output | ("rng",) an sb200_stdrng.
SPECS = [
    ("verify", "verify", True, (), [("in", "pk"), ("in", "u"), ("in", "R"), ("in", "msg"), ("bm",), ("out", 8)]),
    ("verify_double", "verify_double", True, (),
     [("in", "pk"), ("in", "pkp"), ("in", "u"), ("in", "R"), ("in", "Rp"), ("in", "msg"), ("bm",), ("out", 8)]),
    ("verify_vargen", "verify_vargen", True, (),
     [("in", "pk"), ("in", "gen"), ("in", "u"), ("in", "R"), ("in", "msg"), ("bm",), ("out", 8)]),
    ("sign", "sign", True, (), [("in", "sk"), ("in", "msg"), ("in", "nonce"), ("out", 8), ("out", 16), ("out", 8)]),
    ("sign_double", "sign_double", True, (),
     [("in", "sk"), ("in", "msg"), ("in", "nonce"), ("out", 8), ("out", 16), ("out", 16), ("out", 8)]),
    ("sign_vargen", "sign_vargen", True, (),
     [("in", "sk"), ("in", "gen"), ("in", "msg"), ("in", "nonce"), ("out", 8), ("out", 16), ("out", 8)]),
    ("keygen", "keygen", True, (), [("in", "sk"), ("out", 16)]),
    ("keygen_double", "keygen_double", True, (), [("in", "sk"), ("out", 16), ("out", 16)]),
    ("keygen_vargen", "keygen_vargen", True, (), [("in", "sk"), ("in", "gen"), ("out", 16)]),
    ("points_decompress", "points_decompress", True, (), [("in", "pk32"), ("out", 16), ("bm",)]),
    ("points_compress", "points_compress", True, (), [("in", "pk"), ("out", 8)]),
    ("scalars_from_wide", "scalars_from_wide", True, (1,), [("in", "wide"), ("out", 8)]),
    ("stdrng_random", "stdrng_random", True, (0,), [("rng",), ("out", 8)]),
] + [
    (f"sign_stdrng[{s}]", "sign_stdrng", True, (s,),
     [("in", "sk"), ("in", "msg"), ("in", "gen"), ("rng",), ("out", 8), ("out", 16), ("out", 16), ("out", 8)])
    for s in range(3)
] + [
    ("fq_to_mont", "fq_to_mont", True, (), [("in", "msg"), ("out", 8)]),
    ("fq_from_mont", "fq_from_mont", True, (), [("in", "msg"), ("out", 8)]),
    ("verify_bytes", "verify_bytes", True, (), [("in", "pk32"), ("in", "sig64"), ("in", "msg32"), ("bm",), ("bm",)]),
    ("sign_bytes", "sign_bytes", True, (), [("in", "sk"), ("in", "msg32"), ("in", "nonce"), ("out", 16), ("bm",)]),
    ("verify_double_bytes", "verify_double_bytes", True, (),
     [("in", "pk64"), ("in", "sig96"), ("in", "msg32"), ("bm",), ("bm",)]),
    ("verify_vargen_bytes", "verify_vargen_bytes", True, (),
     [("in", "pkg64"), ("in", "sig64"), ("in", "msg32"), ("bm",), ("bm",)]),
    ("sign_double_bytes", "sign_double_bytes", True, (), [("in", "sk"), ("in", "msg32"), ("in", "nonce"), ("out", 24), ("bm",)]),
    ("sign_vargen_bytes", "sign_vargen_bytes", True, (), [("in", "skg64"), ("in", "msg32"), ("in", "nonce"), ("out", 16), ("bm",)]),
] + [
    (f"sign_witness[{s}]", "sign_witness", True, (s,),
     [("in", "sk"), ("in", "msg"), ("in", "nonce"), ("in", "gen"), ("out", 8 * (11, 19, 13)[s])])
    for s in range(3)
] + [
    ("points_check", "points_check", True, (), [("in", "pk"), ("bm",)]),
    ("dbg_verify_ec", "dbg_verify_ec", True, (), [("in", "pk"), ("in", "u"), ("in", "R"), ("in", "c"), ("bm",)]),
    ("dbg_fq", "dbg_fq", False, (0,), [("in", "msg"), ("in", "msg"), ("out", 8)]),
    ("dbg_lattice3", "dbg_lattice3", False, (), [("in", "c"), ("in", "u"), ("out", 32)]),
    ("dbg_fr_mul", "dbg_fr_mul", False, (), [("in", "sk"), ("in", "nonce"), ("out", 8)]),
    ("dbg_hades", "dbg_hades", False, (0,), [("in", "state")]),
    ("dbg_scalar_mul", "dbg_scalar_mul", True, (2,), [("in", "pk"), ("in", "sk"), ("out", 16)]),
]

# Return codes of the default build.  flags: one per bit of FLAG_BITS (None: the call takes no flags); null / mis: one per
# pointer argument, in ABI order (None: not an array); then n = 0 and n = -1.
_ = None
EXPECTED = {
    #                       flags 1    2   4    8    16   64     null                               misaligned
    "verify":              ((OK, OK, ARG, OK, ARG, ARG), (ARG, ARG, ARG, ARG, ARG, OK), (ARG, ARG, ARG, ARG, OK, ARG)),
    "verify_double":       ((OK, OK, ARG, OK, ARG, ARG), (ARG,) * 7 + (OK,), (ARG,) * 6 + (OK, ARG)),
    "verify_vargen":       ((OK, OK, ARG, OK, ARG, ARG), (ARG,) * 6 + (OK,), (ARG,) * 5 + (OK, ARG)),
    "sign":                ((OK, OK, ARG, ARG, OK, ARG), (ARG,) * 5 + (OK,), (ARG,) * 6),
    "sign_double":         ((OK, OK, ARG, ARG, OK, ARG), (ARG,) * 6 + (OK,), (ARG,) * 7),
    "sign_vargen":         ((OK, OK, ARG, ARG, OK, ARG), (ARG,) * 6 + (OK,), (ARG,) * 7),
    "keygen":              ((OK, OK, ARG, ARG, OK, ARG), (ARG, ARG), (ARG, ARG)),
    "keygen_double":       ((OK, OK, ARG, ARG, OK, ARG), (ARG, ARG, ARG), (ARG, ARG, ARG)),
    "keygen_vargen":       ((OK, OK, ARG, ARG, OK, ARG), (ARG, ARG, ARG), (ARG, ARG, ARG)),
    "points_decompress":   ((ARG, OK, ARG, ARG, ARG, ARG), (ARG, ARG, ARG), (ARG, ARG, OK)),
    "points_compress":     ((OK, OK, ARG, ARG, ARG, ARG), (ARG, ARG), (ARG, ARG)),
    "scalars_from_wide":   ((ARG, OK, ARG, ARG, ARG, ARG), (ARG, ARG), (ARG, ARG)),
    "stdrng_random":       ((ARG, OK, ARG, ARG, ARG, ARG), (ARG, ARG), (_, ARG)),
    "sign_stdrng[0]":      ((ARG, OK, ARG, ARG, OK, ARG), (ARG, ARG, OK, ARG, ARG, ARG, OK, OK), (ARG, ARG, OK, _, ARG, ARG, OK, ARG)),
    "sign_stdrng[1]":      ((ARG, OK, ARG, ARG, OK, ARG), (ARG, ARG, OK, ARG, ARG, ARG, ARG, OK), (ARG, ARG, OK, _, ARG, ARG, ARG, ARG)),
    "sign_stdrng[2]":      ((OK, OK, ARG, ARG, OK, ARG), (ARG, ARG, ARG, ARG, ARG, ARG, OK, OK), (ARG, ARG, ARG, _, ARG, ARG, OK, ARG)),
    "fq_to_mont":          ((ARG, OK, ARG, ARG, ARG, ARG), (ARG, ARG), (ARG, ARG)),
    "fq_from_mont":        ((ARG, OK, ARG, ARG, ARG, ARG), (ARG, ARG), (ARG, ARG)),
    "verify_bytes":        ((ARG, OK, ARG, ARG, ARG, ARG), (ARG, ARG, ARG, ARG, OK), (ARG, ARG, ARG, OK, ARG)),
    "sign_bytes":          ((ARG, OK, ARG, ARG, ARG, ARG), (ARG, ARG, ARG, ARG, OK), (ARG, ARG, ARG, ARG, OK)),
    "verify_double_bytes": ((ARG, OK, ARG, ARG, ARG, ARG), (ARG, ARG, ARG, ARG, OK), (ARG, ARG, ARG, OK, ARG)),
    "verify_vargen_bytes": ((ARG, OK, ARG, ARG, ARG, ARG), (ARG, ARG, ARG, ARG, OK), (ARG, ARG, ARG, OK, ARG)),
    "sign_double_bytes":   ((ARG, OK, ARG, ARG, ARG, ARG), (ARG, ARG, ARG, ARG, OK), (ARG, ARG, ARG, ARG, OK)),
    "sign_vargen_bytes":   ((ARG, OK, ARG, ARG, ARG, ARG), (ARG, ARG, ARG, ARG, OK), (ARG, ARG, ARG, ARG, OK)),
    "sign_witness[0]":     ((ARG, OK, ARG, ARG, ARG, ARG), (ARG, ARG, ARG, OK, ARG), (ARG, ARG, ARG, OK, ARG)),
    "sign_witness[1]":     ((ARG, OK, ARG, ARG, ARG, ARG), (ARG, ARG, ARG, OK, ARG), (ARG, ARG, ARG, OK, ARG)),
    "sign_witness[2]":     ((OK, OK, ARG, ARG, ARG, ARG), (ARG,) * 5, (ARG,) * 5),
    "points_check":        ((OK, OK, ARG, ARG, ARG, ARG), (ARG, ARG), (ARG, OK)),
    "dbg_verify_ec":       ((OK, OK, ARG, ARG, ARG, ARG), (ARG,) * 5, (ARG,) * 4 + (OK,)),
    "dbg_fq":              (_, (ARG, OK, ARG), (ARG, ARG, ARG)),
    "dbg_lattice3":        (_, (ARG, ARG, ARG), (ARG, ARG, ARG)),
    "dbg_fr_mul":          (_, (ARG, ARG, ARG), (ARG, ARG, ARG)),
    "dbg_hades":           (_, (ARG,), (ARG,)),
    "dbg_scalar_mul":      ((OK, OK, ARG, ARG, ARG, ARG), (ARG, ARG, ARG), (ARG, ARG, ARG)),
}
EXPECTED_N0, EXPECTED_NEG = OK, ARG

# kernel launches per pipeline chunk (per call with device pointers)
LAUNCHES = {
    "verify": 2, "verify_double": 2, "verify_vargen": 2,                        # challenge, curve
    "verify_bytes": 3, "verify_double_bytes": 3, "verify_vargen_bytes": 3,      # decode, challenge, curve
    "sign_stdrng[0]": 2, "sign_stdrng[1]": 2, "sign_stdrng[2]": 2,              # draws, sign
    **{k: 1 for k in ("sign", "sign_double", "sign_vargen", "keygen", "keygen_double", "keygen_vargen", "points_decompress",
                      "points_compress", "scalars_from_wide", "stdrng_random", "fq_to_mont", "fq_from_mont", "sign_bytes",
                      "sign_double_bytes", "sign_vargen_bytes", "sign_witness[0]", "sign_witness[1]", "sign_witness[2]",
                      "points_check", "dbg_verify_ec", "dbg_fq", "dbg_lattice3", "dbg_fr_mul", "dbg_hades", "dbg_scalar_mul")},
}
SENTINEL = 0xA5A5A5A5


def test_tables_cover_every_compute_entry_point():
    from schnorr_b200 import _lib
    compute = {s[len("sb200_"):] for s in _lib.EXPORTED_SYMBOLS} - {
        "init", "init_ex", "default_params", "get_params", "params_check", "dbg_hades_tables", "destroy", "strerror",
        "last_error", "device_count", "set_stream", "launch_count", "host_alloc", "host_free"}
    assert {s[1] for s in SPECS} == compute
    assert [s[0] for s in SPECS] == list(EXPECTED) and set(LAUNCHES) == set(EXPECTED)
    for sid, _n, has_flags, _i, args in SPECS:
        flags, null, mis = EXPECTED[sid]
        assert (flags is None) == (not has_flags) and len(null) == len(mis) == len(args), sid


@pytest.fixture
def base(engine):
    """32 well-formed tuples of every input array (keys and signatures from the library, projective points with Z = 1)"""
    rs = np.random.RandomState(7)

    def sc(bits):
        a = rs.randint(0, 1 << 32, size=(32, 8), dtype=np.uint64).astype(np.uint32)
        a[:, 7] &= (1 << bits) - 1
        return a

    sk, nonce, msg, c = sc(27), sc(27), sc(30), sc(27)
    one = np.tile(V.mont(1), (32, 1))
    proj = lambda p: np.ascontiguousarray(np.concatenate([p, one], axis=1))
    pk, pkp = engine.keygen_double(sk)
    gen = pk
    u, R, Rp, _c = engine.sign_double(sk, msg, nonce)
    pk32, pkp32 = engine.points_compress(pk), engine.points_compress(pkp)
    R32, Rp32 = engine.points_compress(R), engine.points_compress(Rp)
    state = np.concatenate([msg, sk, nonce, c, msg], axis=1)
    wide = np.concatenate([sk, msg], axis=1)
    b = dict(sk=sk, nonce=nonce, msg=msg, c=c, u=u, pk=proj(pk), pkp=proj(pkp), gen=proj(gen), R=proj(R), Rp=proj(Rp),
             pk32=pk32, msg32=sk, sig64=np.concatenate([u, R32], axis=1), sig96=np.concatenate([u, R32, Rp32], axis=1),
             pk64=np.concatenate([pk32, pkp32], axis=1), pkg64=np.concatenate([pk32, pk32], axis=1),
             skg64=np.concatenate([sk, pk32], axis=1), state=state, wide=wide)
    return {k: np.ascontiguousarray(v, dtype=np.uint32) for k, v in b.items()}


class Call:
    """one entry point's buffers over n tuples, on the host (64-byte aligned numpy) or on the device (torch)"""

    def __init__(self, engine, spec, base, n, device=False):
        self.engine, self.spec, self.n, self.device = engine, spec, n, device
        self.arrays = []
        for a in spec[4]:
            if a[0] == "in":
                self.arrays.append(np.tile(base[a[1]], (-(-n // 32), 1))[:n])
            elif a[0] == "out":
                self.arrays.append(np.full((n, a[1]), SENTINEL, np.uint32))
            elif a[0] == "bm":
                self.arrays.append(np.full(((n + 31) // 32,), SENTINEL, np.uint32))
            else:
                self.arrays.append(None)
        self.reset()

    def reset(self):
        from schnorr_b200 import _lib
        self.bufs = []
        for a in self.arrays:
            if a is None:
                self.bufs.append(None)
            elif self.device:
                import torch
                self.bufs.append(torch.from_numpy(a.view(np.int32).copy()).to("cuda:0"))
            else:
                buf = _lib.aligned_empty((a.size + 4,))
                buf[:a.size] = a.reshape(-1)
                self.bufs.append(buf)
        self.rng = _lib.StdRngPos.of([0x01010101 * (k + 1) for k in range(8)], 1 << 40)

    def ptr(self, k):
        b = self.bufs[k]
        if b is None:
            return ctypes.byref(self.rng)
        return ctypes.c_void_p(b.data_ptr() if self.device else b.ctypes.data)

    def __call__(self, flags=0, n=None, null=None, mis=None):
        _sid, name, has_flags, ints, args = self.spec
        ptrs = [self.ptr(k) for k in range(len(args))]
        if null is not None:
            ptrs[null] = None
        if mis is not None:
            ptrs[mis] = ctypes.c_void_p(self.bufs[mis].ctypes.data + 4)
        lead = [self.engine._h, self.n if n is None else n] + ([flags] if has_flags else []) + list(ints)
        before = self.engine.launch_count
        rc = getattr(self.engine._lib, "sb200_" + name)(*lead, *ptrs)
        if self.device:
            import torch
            torch.cuda.synchronize()
        return rc, self.engine.launch_count - before

    def outputs(self):
        """the arrays a call may write, as they are now"""
        return [b.cpu().numpy().view(np.uint32).reshape(-1) if self.device else b[:-4].copy()
                for a, b in zip(self.spec[4], self.bufs) if a[0] in ("out", "bm") or a == ("in", "state")]

    def initial_outputs(self):
        return [x.reshape(-1) for a, x in zip(self.spec[4], self.arrays) if a[0] in ("out", "bm") or a == ("in", "state")]


def _cases(sid, nargs, has_flags):
    """(label, call kwargs, expected rc) of every variation of one entry point's valid call"""
    flags, null, mis = EXPECTED[sid]
    out = []
    if has_flags:
        out += [(f"flag {f}", dict(flags=f), rc) for f, rc in zip(FLAG_BITS, flags)]
    out += [(f"null arg {k}", dict(null=k), null[k]) for k in range(nargs)]
    out += [(f"misaligned arg {k}", dict(mis=k), mis[k]) for k in range(nargs) if mis[k] is not None]
    out += [("n = 0", dict(n=0), EXPECTED_N0), ("n = -1", dict(n=-1), EXPECTED_NEG)]
    return out


@pytest.mark.parametrize("spec", SPECS, ids=[s[0] for s in SPECS])
def test_accept_reject_matrix_and_the_context_stays_usable(engine, base, spec):
    sid, _name, has_flags, _ints, args = spec
    ref = Call(engine, spec, base, N_SMALL)
    assert ref() == (OK, LAUNCHES[sid])
    want = ref.outputs()
    got = {}
    for label, kw, rc_want in _cases(sid, len(args), has_flags):
        call = Call(engine, spec, base, N_SMALL, device=kw.get("flags") == 2)  # device pointers need device buffers
        rc, launched = call(**kw)
        got[label] = rc
        if rc == OK:
            assert launched == (0 if kw.get("n") == 0 else LAUNCHES[sid]), label
        else:
            assert launched == 0, label
        if rc != OK or kw.get("n") == 0:
            assert all((x == y).all() for x, y in zip(call.outputs(), call.initial_outputs())), f"{label}: outputs written"
            assert call.rng.word_pos == 1 << 40, f"{label}: StdRng position moved"
    assert got == {label: rc for label, _kw, rc in _cases(sid, len(args), has_flags)}
    again = Call(engine, spec, base, N_SMALL)
    assert again() == (OK, LAUNCHES[sid])
    assert all((x == y).all() for x, y in zip(again.outputs(), want)), "the valid call after the rejections differs"


@pytest.mark.parametrize("spec", SPECS, ids=[s[0] for s in SPECS])
def test_launch_counts_per_chunk(engine, base, spec):
    """also with each optional output left null: a split verification without c_out hands its challenges over in scratch,
    a byte-level verification without `invalid` keeps its invalid bitmap there"""
    sid, _name, has_flags, _ints, args = spec
    chunks = host_chunks(N_CHUNKS)
    assert len(chunks) > 1
    optional = [k for k, a in enumerate(args) if a[0] in ("out", "bm") and EXPECTED[sid][1][k] == OK]
    for kw in [{}] + [dict(null=k) for k in optional]:
        assert Call(engine, spec, base, N_SMALL)(**kw) == (OK, LAUNCHES[sid]), kw
        assert Call(engine, spec, base, N_CHUNKS)(**kw) == (OK, LAUNCHES[sid] * len(chunks)), kw
        if has_flags:  # the debug calls without flags take host buffers only
            assert Call(engine, spec, base, N_SMALL, device=True)(flags=2, **kw) == (OK, LAUNCHES[sid]), kw
