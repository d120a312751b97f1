"""schnorr_b200: B200-native batch engine for dusk-schnorr's sign / verify hot path.

Layout: `csrc/` holds the CUDA kernels and the C ABI (`include/schnorr_b200.h`);
`_lib.py` binds the ABI with ctypes; `api.py` mirrors the reference crate's types
(SecretKey, PublicKey, Signature, the Double and VarGen variants) on top of it.
There is no CPU fallback anywhere in this package.
"""
from ._lib import (ARK_CUMSUM, ARK_ENV, ARK_PLAIN, CHECK_POINTS, DEVICE_PTRS, POINTS_AFFINE, POINTS_PROJECTIVE, SIGN_OBLIVIOUS,  # noqa: F401
                   VERIFY_DUAL_PIPE, Engine, KeySet, Params, PinnedBuffer, SchnorrB200Error, default_params, load_library)
