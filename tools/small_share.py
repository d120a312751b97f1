import os, sys, time, json
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
from schnorr_b200 import POINTS_AFFINE, Engine, PinnedBuffer
lg = int(sys.argv[1]) if len(sys.argv) > 1 else 19
n = 1 << lg
rs = np.random.RandomState(3)
def sc(bits):
    a = rs.randint(0, 1 << 32, size=(n, 8), dtype=np.uint64).astype(np.uint32); a[:, 7] &= (1 << bits) - 1; return a
sk, nonce, msg = sc(27), sc(27), sc(30)
e = Engine([0])
pk = e.keygen(sk); u, R, _ = e.sign(sk, msg, nonce)
keep = [PinnedBuffer(s) for s in ((n, 16), (n, 8), (n, 16), (n, 8), ((n + 31) // 32,))]
bufs = [b.array for b in keep]
for dst, src in zip(bufs[:4], (pk, u, R, msg)): dst[...] = src
P = lambda a: a.ctypes.data
call = lambda: e.call("verify", n, POINTS_AFFINE, P(bufs[0]), P(bufs[1]), P(bufs[2]), P(bufs[3]), P(bufs[4]), None)
call(); call()
t0 = time.perf_counter()
for _ in range(10): call()
dt = (time.perf_counter() - t0) / 10
ok = np.unpackbits(bufs[4].view(np.uint8), bitorder="little")[:n]
print(json.dumps({"mode": os.environ.get("SB200_CURVE_PERSISTENT", "auto"), "n": n, "ms": dt * 1e3, "M_per_s": n / dt / 1e6, "all_true": bool(ok.all())}))
