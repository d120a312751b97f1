#!/usr/bin/env python3
"""bench.py -- the measurements of the sign/verify hot path.

    python bench.py --gpus N --steps K --warmup W            (N>1: under torchrun, one rank per GPU)
    python bench.py --impl reference --gpus N --steps K --warmup W
    python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR

`--steps K` is the number of timed steps of every timed loop (the top-level record, `e2e`, each of `configs` and
`strong_scaling`).  `--dump-outputs DIR` writes what the top-level record's last timed step computed, the verdict of
every tuple (rank 0's shard when N > 1), to DIR/verify_ok.npy (float32, 1.0 = the signature verifies); the inputs are
seeded, so two builds run with the same arguments can be compared output for output.  bench.py writes nothing into
the source tree, which may be read-only.

TOP-LEVEL RECORD (the driver's contract; config.workload): single-key `PublicKey::verify`
(/root/reference/src/keys/public.rs:121-130) over 2^22 (message, key, signature) tuples PER GPU (weak scaling:
tuples are independent, sharded by index, no collective), 10 % of the signatures corrupted.  A "step" = one pass of
the verify path over the whole batch.  Inputs are synthetic: seeded keys / messages / nonces, signed with the
engine's own batch signer (whose parity with the oracle is what tests/ establish).

  value        verifies/s, inputs resident in HBM (DEVICE_PTRS call, CUDA events on the launching stream)
  e2e          verifies/s through the host-buffer C-ABI call (pinned host inputs; H2D + kernels + D2H of the verdict
               bitmap inside the timed region)
  roofline     IMAD.WIDE issue roofline (the path is integer-multiply bound; HBM share reported too); `peak` is the
               measured rate (IMAD_PEAK.json), `peak_nominal` / `frac_nominal` the 32/clk/SM figure beside it
  cpu_baseline oracle/ref_cpu.c (C restatement of the reference's algorithm, all host cores) on a bounded prefix of
               the same batch; its verdicts are compared with the GPU's.

`configs` -- one first-class record (value, e2e, roofline, cpu_baseline, a content check against the CPU
restatement) for every configuration BASELINE.json names:
  c0_single_tuple_cpu     one sign + one verify, seed 2321, one core  (/root/reference/tests/schnorr.rs:15-25)
  c1_verify_2_16          single-key verify, 2^16 valid signatures
  c2_verify_double_2_20   PublicKeyDouble::verify with real (pk, pk', R, R')   (public.rs:222-244)
  c3_sign_2_20 / _2_22    SecretKey::sign with nonces from the seeded ChaCha12 stream (secret.rs:150-168)
  c4_verify_vargen_2_22   PublicKeyVarGen::verify, per-key generators, 10 % corrupted in four ways (public.rs:401-415)
  verify_bytes_2_20       the wire-level call: PublicKey / Signature / BlsScalar::from_bytes on the device + verify
plus `e2e_typed` (the typed C++ host API with pageable memory, tools/bench_typed.cpp) and, when N > 1,
`strong_scaling` (ONE context over all N devices splitting a single 2^22 batch from host buffers).

`--impl reference` times the CPU restatement alone (the Rust crate cannot be built in this image).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # no __pycache__ in the source tree

LOG2_BATCH = 22
METRIC = "verifies_per_s"
UNIT = "verifies/s"
# 32x32->64 limb products one tuple executes in each kernel, counted by the instrumented host build of the same
# code (tools/op_counts.py; tests/test_op_counts.py keeps the file honest).
OPCOUNT_FILE = os.path.join(ROOT, "profiles", "op_counts.json")
IMAD_PEAK_FILE = os.path.join(ROOT, "IMAD_PEAK.json")


def synth_scalars(rs, n, top_bits):
    a = rs.randint(0, 1 << 32, size=(n, 8), dtype=np.uint64).astype(np.uint32)
    a[:, 7] &= (1 << top_bits) - 1
    return a


def make_inputs(n, seed):
    """sk, nonce < 2^251 < r (canonical scalars); msg < 2^254 < q (Montgomery limbs of some field element)."""
    rs = np.random.RandomState(seed)
    return synth_scalars(rs, n, 27), synth_scalars(rs, n, 27), synth_scalars(rs, n, 30)


def corrupt_mask(n):
    return (np.arange(n, dtype=np.int64) * 2654435761 % 10) == 0  # deterministic ~10 %


DUMP_BYTES = 64 * 10**6  # --dump-outputs writes at most this much in all
DUMP_SAMPLE, DUMP_SAMPLE_SEED = 1 << 22, 0xD0  # 2^22 x (float32 value + float64 index) = 50 MB


def dump_outputs(out_dir, name, values):
    """values (one per tuple) -> out_dir/<name>.npy as float32.  A batch too large for DUMP_BYTES is replaced by a fixed,
    seeded sample of DUMP_SAMPLE tuples, whose indices go to out_dir/<name>_index.npy (float64, exact below 2^53)."""
    os.makedirs(out_dir, exist_ok=True)
    values = np.asarray(values, dtype=np.float32)
    if values.nbytes > DUMP_BYTES:
        idx = np.sort(np.random.RandomState(DUMP_SAMPLE_SEED).choice(len(values), DUMP_SAMPLE, replace=False))
        np.save(os.path.join(out_dir, name + "_index.npy"), idx.astype(np.float64))
        values = values[idx]
    np.save(os.path.join(out_dir, name + ".npy"), values)


# ---- rand 0.8 StdRng (ChaCha12) over whole blocks, vectorised: block i of the stream = the 64 bytes that the i-th
# `JubJubScalar::random` of a signing loop consumes (/root/reference/src/keys/secret.rs:155).  Host side, as in the
# reference; the reduction mod r (from_bytes_wide) runs on the device (sb200_scalars_from_wide).
def seed_from_u64(state):
    out = []
    for _ in range(8):
        state = (state * 6364136223846793005 + 11634580027462260723) & ((1 << 64) - 1)
        xs = (((state >> 18) ^ state) >> 27) & 0xFFFFFFFF
        rot = state >> 59
        out.append(((xs >> rot) | (xs << ((32 - rot) & 31))) & 0xFFFFFFFF)
    return out


def chacha12_blocks(key_words, first, count):
    ctr = np.arange(first, first + count, dtype=np.uint64)
    st = [np.full(count, c, np.uint32) for c in (0x61707865, 0x3320646E, 0x79622D32, 0x6B206574)]
    st += [np.full(count, k, np.uint32) for k in key_words]
    st += [(ctr & 0xFFFFFFFF).astype(np.uint32), (ctr >> np.uint64(32)).astype(np.uint32), np.zeros(count, np.uint32), np.zeros(count, np.uint32)]
    x = [s.copy() for s in st]
    rotl = lambda v, r: (v << np.uint32(r)) | (v >> np.uint32(32 - r))

    def qr(a, b, c, d):
        x[a] += x[b]; x[d] = rotl(x[d] ^ x[a], 16)
        x[c] += x[d]; x[b] = rotl(x[b] ^ x[c], 12)
        x[a] += x[b]; x[d] = rotl(x[d] ^ x[a], 8)
        x[c] += x[d]; x[b] = rotl(x[b] ^ x[c], 7)

    for _ in range(6):
        qr(0, 4, 8, 12); qr(1, 5, 9, 13); qr(2, 6, 10, 14); qr(3, 7, 11, 15)
        qr(0, 5, 10, 15); qr(1, 6, 11, 12); qr(2, 7, 8, 13); qr(3, 4, 9, 14)
    return np.stack([a + b for a, b in zip(x, st)], axis=1)  # [count, 16] u32 = 64 little-endian bytes per block


def stdrng_nonces(eng, seed, n):
    """nonce i = JubJubScalar::from_bytes_wide(block i of StdRng::seed_from_u64(seed))"""
    key = seed_from_u64(seed)
    out = np.empty((n, 8), np.uint32)
    step = 1 << 20
    for lo in range(0, n, step):
        blocks = chacha12_blocks(key, lo, min(step, n - lo))
        out[lo:lo + len(blocks)] = eng.scalars_from_wide(blocks.view(np.uint8), 0)
    return out


class ClockSampler(threading.Thread):
    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz, self.power = index, [], set(), False, None, []
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if not self.nv:
            return
        nv = self.nv
        names = {"GpuIdle": "gpu_idle", "SwPowerCap": "sw_power_cap", "HwSlowdown": "hw_slowdown",
                 "SwThermalSlowdown": "sw_thermal_slowdown", "HwThermalSlowdown": "hw_thermal_slowdown",
                 "HwPowerBrakeSlowdown": "hw_power_brake", "ApplicationsClocksSetting": "applications_clocks_setting",
                 "SyncBoost": "sync_boost", "DisplayClockSetting": "display_clock_setting"}
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                self.power.append(nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0)
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, v in names.items():
                    bit = getattr(nv, "nvmlClocksThrottleReason" + k, 0)
                    if bit and (r & bit):
                        self.reasons.add(v)
            except Exception:
                pass
            time.sleep(0.05)

    def result(self):
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(x for x in self.reasons if x != "gpu_idle"), "samples": len(s),
                "power_w_max": max(self.power) if self.power else None}


def ncu_traffic(key, n):
    """dram__bytes_read.sum + dram__bytes_write.sum of the op's launches from the committed `ncu --set full` capture
    (profiles/ncu_traffic.json, written by tools/ncu_traffic.py), scaled to this launch's tuple count; None if absent."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))[key]
        return (t["dram_bytes_read"] + t["dram_bytes_write"]) * n / t["tuples"]
    except Exception:
        return None


def roofline(op_key, n, ms, bytes_io, traffic_key=None):
    """IMAD.WIDE roofline of one op: executed limb products per tuple (profiles/op_counts.json) x tuples / time."""
    try:
        peak = json.load(open(IMAD_PEAK_FILE))
        ops = json.load(open(OPCOUNT_FILE))[op_key]
        wide = ops["imad_wide_per_tuple"]
        achieved = n * wide / (ms * 1e-3) / 1e12
        hbm_peak = 6650.0
        mp = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(mp):
            hbm_peak = json.load(open(mp))["hbm_gbs"]
        hbm = bytes_io / (ms * 1e-3) / 1e9
        issue = None
        try:  # issue-slot model (DESIGN.md 4.0): executed warp instructions per tuple from the committed ncu captures
            ic = json.load(open(os.path.join(ROOT, "profiles", "inst_counts.json")))[op_key]
            im = json.load(open(os.path.join(ROOT, "profiles", "issue_model.json")))
            inst = ic["warp_inst_per_tuple"]
            a_w, b_o = im["cycles_per_wide"], im["cycles_per_other"]
            smsp_cycles_per_s = im["sm_subpartitions"] * im["sm_hz"]
            need = (a_w * wide + b_o * (inst - wide)) * n / 32.0  # sub-partition cycles the model asks for this launch
            issue = {"model": f"{a_w} cycles per IMAD.WIDE + {b_o} per other warp instruction on one SM sub-partition "
                              "(fit of tools/issue_mix.cu, profiles/issue_mix_r02.json; accuracy about 10 %)",
                     "warp_inst_per_tuple": inst, "wide_per_tuple": wide, "inst_source": ic["source"],
                     "predicted_ms": need / smsp_cycles_per_s * 1e3, "measured_ms": ms,
                     "predicted_over_measured": need / smsp_cycles_per_s * 1e3 / ms}
        except Exception:
            issue = None
        return {"bound": "imad", "issue_model": issue, "achieved": achieved, "peak": peak["imad_wide_per_s"] / 1e12, "unit": "T IMAD.WIDE/s",
                "frac": achieved / (peak["imad_wide_per_s"] / 1e12),
                "peak_nominal": peak["nominal_per_s"] / 1e12, "frac_nominal": achieved / (peak["nominal_per_s"] / 1e12),
                "traffic": ncu_traffic(traffic_key, n) if traffic_key else None,
                "peak_source": "IMAD_PEAK.json: tools/imad_peak.cu on this pool's B200, 1 s launches, SM clock measured in the kernel "
                               f"({peak.get('sm_mhz_in_kernel')} MHz); nominal = 32/clk/SM x 148 SMs x 1965 MHz",
                "work": f"{wide} IMAD.WIDE.U32 per tuple ({ops.get('fq_mul')} fq_mul, {ops.get('fq_sqr')} fq_sqr, "
                        f"{ops.get('fq_dot5', 0)} fq_dot5, {ops.get('fr_mont_mul', 0)} fr_mont_mul)" + (f"; {ops['note']}" if "note" in ops else ""),
                "hbm": {"achieved_gbs": hbm, "peak_gbs": hbm_peak, "frac": hbm / hbm_peak}}
    except Exception as ex:  # pragma: no cover
        return {"bound": "imad", "error": repr(ex)}


def cpu_reference_arm(args):
    """The reference's CPU implementation of the path = oracle/ref_cpu.c, all host threads."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import ref_cpu
    cores = os.cpu_count() or 1
    n = args.ref_sample or 2048 * cores
    sk, nonce, msg = make_inputs(n, 0xC1)
    pk = ref_cpu.keygen(sk)
    u, R, _ = ref_cpu.sign(sk, msg, nonce)
    bad = corrupt_mask(n)
    u[bad, 0] ^= 1
    for _ in range(args.warmup):
        ref_cpu.verify(pk[:256 * cores], u[:256 * cores], R[:256 * cores], msg[:256 * cores])
    t0 = time.perf_counter()
    for _ in range(args.steps):
        ok, _ = ref_cpu.verify(pk, u, R, msg)
    dt = (time.perf_counter() - t0) / args.steps
    assert (ok == ~bad).all(), "CPU restatement verdicts are wrong"
    val = n / dt
    sample = f"{n} tuples/step (prefix of the 2^{LOG2_BATCH} workload), {cores} pthreads"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u64", "data": "synthetic",
        "config": {"workload": f"single-key PublicKey::verify, 10% corrupted, CPU restatement of dusk-schnorr's algorithm "
                               f"(the Rust crate cannot be built in this image), bounded sample of {n} tuples per step"},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--log2-batch", type=int, default=LOG2_BATCH)
    ap.add_argument("--ref-sample", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="top-level record only (no `configs`, typed, strong scaling)")
    ap.add_argument("--only", default="", help="comma-separated config names to run (development aid)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the top-level record's per-tuple verdicts of its last timed step to DIR/verify_ok.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 0)
    if args.impl == "reference":
        return cpu_reference_arm(args)

    import torch
    import torch.distributed as dist
    from schnorr_b200 import DEVICE_PTRS, POINTS_AFFINE, Engine, PinnedBuffer

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        # NCCL_DEBUG=VERSION (some boxes export it) makes NCCL print its banner on stdout, next to the one JSON line
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    torch.cuda.set_device(local)
    dev = torch.device(f"cuda:{local}")
    eng = Engine([local])  # raises without a GPU: there is no CPU fallback
    n = 1 << args.log2_batch
    cores = os.cpu_count() or 1
    stream = torch.cuda.current_stream()
    eng.set_stream(stream.cuda_stream)
    P = lambda t: t.data_ptr() if hasattr(t, "data_ptr") else t.ctypes.data
    npv = lambda t: t.numpy().view(np.uint32)
    ref_cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import ref_cpu

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def to_dev(a):
        return torch.from_numpy(np.ascontiguousarray(a).view(np.int32)).to(dev)

    def pinned(a):
        """a copy of `a` in page-locked host memory (torch's allocator: freed with the tensor)"""
        t = torch.empty(a.shape, dtype=torch.int32 if a.dtype == np.uint32 else torch.uint8, pin_memory=True)
        t.numpy().view(a.dtype)[...] = a
        return t

    def unpack(bm, cnt):
        a = bm.cpu().numpy() if hasattr(bm, "cpu") else bm
        return np.unpackbits(np.ascontiguousarray(a).view(np.uint8), bitorder="little")[:cnt].astype(bool)

    def time_device(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = eng.launch_count
        e0.record(stream)
        for _ in range(steps):
            fn()
        e1.record(stream)
        barrier()
        return max_over_ranks(e0.elapsed_time(e1) / steps), eng.launch_count - l0

    def time_host(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            fn()
        torch.cuda.synchronize()
        return max_over_ranks((time.perf_counter() - t0) / steps)

    # ---- top-level record: single-key verify, 2^22 per GPU, 10 % corrupted --------------------------------------
    sk, nonce, msg = make_inputs(n, 0xC1 + rank)
    pk = eng.keygen(sk)
    u, R, c_sign = eng.sign(sk, msg, nonce)
    bad = corrupt_mask(n)
    u[bad, 0] ^= 1  # still canonical (< r): flips the lowest bit
    h_pk, h_u, h_R, h_msg = pinned(pk), pinned(u), pinned(R), pinned(msg)
    h_bm = torch.zeros((n + 31) // 32, dtype=torch.int32).pin_memory()
    d_pk, d_u, d_R, d_msg = (t.to(dev) for t in (h_pk, h_u, h_R, h_msg))
    d_bm = torch.zeros((n + 31) // 32, dtype=torch.int32, device=dev)
    fl = POINTS_AFFINE | DEVICE_PTRS

    sampler = ClockSampler(local)
    sampler.start()
    ms_step, launches = time_device(lambda: eng.call("verify", n, fl, P(d_pk), P(d_u), P(d_R), P(d_msg), P(d_bm), None),
                                    args.steps, args.warmup)
    sampler.stop_flag = True
    verdict = unpack(d_bm, n)
    assert (verdict == ~bad).all(), "GPU verdicts wrong: valid signatures must verify, corrupted ones must not"
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, "verify_ok", verdict)
    value = world * n / (ms_step * 1e-3)
    e2e_s = time_host(lambda: eng.call("verify", n, POINTS_AFFINE, P(h_pk), P(h_u), P(h_R), P(h_msg), P(h_bm), None),
                      args.steps, min(args.warmup, 2))
    assert (unpack(npv(h_bm), n) == ~bad).all()
    e2e = world * n / e2e_s
    h2d = n * (16 + 8 + 16 + 8) * 4
    d2h = ((n + 31) // 32) * 4
    roof = roofline("verify_affine", n, ms_step, h2d + d2h, "verify_affine")
    cpu = None
    if ref_cpu:
        ns = args.ref_sample or 1024 * cores
        t0 = time.perf_counter()
        okc, _ = ref_cpu.verify(pk[:ns], u[:ns], R[:ns], msg[:ns])
        dt = time.perf_counter() - t0
        assert (okc == verdict[:ns]).all(), "GPU and CPU-restatement verdicts differ"
        cpu = {"value": ns / dt, "unit": UNIT, "cores": cores, "kind": "port",
               "sample": f"first {ns} tuples of the batch, {cores} pthreads; verdicts identical to the GPU's"}

    # ---- first-class records for the other BASELINE configurations ---------------------------------------------------
    configs = {}
    only = set(x for x in args.only.split(",") if x)
    want = lambda name: not args.no_extras and (not only or name in only)
    ksteps, kwarm = args.steps, max(1, min(args.warmup, 2))

    def record(name, workload, cnt, unit, op_key, dev_call, host_call, h2d_b, d2h_b, check, cpu_fn=None, traffic_key=None):
        ms, _ = time_device(dev_call, ksteps, kwarm)
        s = time_host(host_call, ksteps, 1)
        checked = check()
        rec = {"workload": workload, "n_per_gpu": cnt, "value": world * cnt / (ms * 1e-3), "unit": unit, "ms_per_step": ms,
               "e2e": {"value": world * cnt / s, "unit": unit, "h2d_bytes_per_step": h2d_b, "d2h_bytes_per_step": d2h_b},
               "roofline": roofline(op_key, cnt, ms, h2d_b + d2h_b, traffic_key), "checked": checked, "cpu_baseline": None}
        if ref_cpu and cpu_fn:
            ns = min(cnt, args.ref_sample or 512 * cores)
            t0 = time.perf_counter()
            note = cpu_fn(ns)
            dt = time.perf_counter() - t0
            rec["cpu_baseline"] = {"value": ns / dt, "unit": unit, "cores": cores, "kind": "port",
                                   "sample": f"first {ns} tuples, {cores} pthreads; {note}"}
        configs[name] = rec

    if want("c0_single_tuple_cpu") and ref_cpu:
        # /root/reference/tests/schnorr.rs:15-25 on ONE core: StdRng::seed_from_u64(2321); sk, message, sign (one nonce draw), verify
        import schnorr_oracle as o
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import vectors as V
        rng = o.StdRng.seed_from_u64(2321)
        sk0, m0, n0 = V.scalars([rng.random_fr()]), V.fqs([rng.random_fq()]), V.scalars([rng.random_fr()])
        pk0 = ref_cpu.keygen(sk0, threads=1)
        reps = 200
        t0 = time.perf_counter()
        for _ in range(reps):
            u0, R0, _ = ref_cpu.sign(sk0, m0, n0, threads=1)
        t_sign = (time.perf_counter() - t0) / reps
        t0 = time.perf_counter()
        for _ in range(reps):
            ok0, _ = ref_cpu.verify(pk0, u0, R0, m0, threads=1)
        t_ver = (time.perf_counter() - t0) / reps
        gu, gR, _ = eng.sign(sk0, m0, n0)
        gok, _ = eng.verify(eng.keygen(sk0), gu, gR, m0)
        t0 = time.perf_counter()
        for _ in range(20):
            eng.sign(sk0, m0, n0)
        g_sign = (time.perf_counter() - t0) / 20
        t0 = time.perf_counter()
        for _ in range(20):
            eng.verify(pk0, gu, gR, m0, want_c=False)
        g_ver = (time.perf_counter() - t0) / 20
        assert ok0.all() and gok.all() and (gu == u0).all() and (gR == R0).all()
        configs["c0_single_tuple_cpu"] = {
            "workload": "reference test recipe (tests/schnorr.rs:15-25, seed 2321): one sign + one verify of one Fq message, CPU restatement on ONE core",
            "cpu_sign_us": t_sign * 1e6, "cpu_verify_us": t_ver * 1e6, "cpu_signs_per_s": 1 / t_sign, "cpu_verifies_per_s": 1 / t_ver,
            "gpu_single_tuple_sign_us": g_sign * 1e6, "gpu_single_tuple_verify_us": g_ver * 1e6,
            "checked": "signature bytes of the GPU and the CPU restatement identical; both verify it",
            "note": "a batch of one is latency-bound on the GPU (two launches + copies); the engine exists for batches"}

    if want("c1_verify_2_16"):
        m = 1 << 16
        s1, n1, m1 = make_inputs(m, 0x1C1 + rank)
        p1 = eng.keygen(s1)
        u1, R1, _ = eng.sign(s1, m1, n1)
        hp = [pinned(a) for a in (p1, u1, R1, m1)]
        dp = [t.to(dev) for t in hp]
        hb, db = torch.zeros(m // 32, dtype=torch.int32).pin_memory(), torch.zeros(m // 32, dtype=torch.int32, device=dev)
        def chk():
            assert unpack(db, m).all() and unpack(npv(hb), m).all()
            return "all 2^16 verdicts true (device-resident and host-buffer calls)"
        def cpu_fn(ns):
            okc, _ = ref_cpu.verify(p1[:ns], u1[:ns], R1[:ns], m1[:ns])
            assert okc.all()
            return "verdicts identical"
        record("c1_verify_2_16", "single-key PublicKey::verify, 2^16 valid signatures, affine Montgomery inputs", m, UNIT, "verify_affine",
               lambda: eng.call("verify", m, fl, *[P(t) for t in dp], P(db), None),
               lambda: eng.call("verify", m, POINTS_AFFINE, *[P(t) for t in hp], P(hb), None), m * 192, m // 8, chk, cpu_fn)

    if want("c2_verify_double_2_20"):
        m = min(n, 1 << 20)
        s2, n2, m2 = make_inputs(m, 0xC2 + rank)
        p2, p2p = eng.keygen_double(s2)
        u2, R2, R2p, _ = eng.sign_double(s2, m2, n2)
        bad2 = corrupt_mask(m)
        mode = np.arange(m) % 3
        u2[bad2 & (mode == 0), 0] ^= 1
        sel = bad2 & (mode == 1); R2p[sel] = np.roll(R2p, -1, axis=0)[sel]   # another tuple's R'
        sel = bad2 & (mode == 2); p2p[sel] = np.roll(p2p, -1, axis=0)[sel]   # another tuple's pk'
        arrs = (p2, p2p, u2, R2, R2p, m2)
        hp = [pinned(a) for a in arrs]
        dp = [t.to(dev) for t in hp]
        hb, db = torch.zeros(m // 32, dtype=torch.int32).pin_memory(), torch.zeros(m // 32, dtype=torch.int32, device=dev)
        def chk():
            assert (unpack(db, m) == ~bad2).all() and (unpack(npv(hb), m) == ~bad2).all()
            return "verdict == not corrupted for all tuples (10 % corrupted: u, R', pk')"
        def cpu_fn(ns):
            okc, _ = ref_cpu.verify_double(*[a[:ns] for a in arrs])
            assert (okc == ~bad2[:ns]).all()
            return "verdicts identical to the GPU's"
        record("c2_verify_double_2_20", "PublicKeyDouble::verify, 2^20 tuples with real (pk, pk', R, R'), 10% corrupted", m, UNIT,
               "verify_double_affine", lambda: eng.call("verify_double", m, fl, *[P(t) for t in dp], P(db), None),
               lambda: eng.call("verify_double", m, POINTS_AFFINE, *[P(t) for t in hp], P(hb), None), m * 352, m // 8, chk, cpu_fn)
        del hp, dp

    for lg in (20, 22):
        name = f"c3_sign_2_{lg}"
        if not want(name) or (1 << lg) > n:
            continue
        m = 1 << lg
        s3, _, m3 = make_inputs(m, 0xC3 + rank)
        n3 = stdrng_nonces(eng, 0xC3 + rank, m)  # the seeded ChaCha12 stream, one block per signature
        hp = [pinned(a) for a in (s3, m3, n3)]
        dp = [t.to(dev) for t in hp]
        ho = [torch.empty((m, k), dtype=torch.int32).pin_memory() for k in (8, 16, 8)]
        do = [torch.empty((m, k), dtype=torch.int32, device=dev) for k in (8, 16, 8)]
        def chk():
            a, b = [t.cpu().numpy().view(np.uint32) for t in do], [npv(t) for t in ho]
            assert all((x == y).all() for x, y in zip(a, b)), "device-resident and host-buffer signatures differ"
            ok3, c3 = eng.verify(eng.keygen(s3[:4096]), b[0][:4096], b[1][:4096], m3[:4096])
            assert ok3.all() and (c3 == b[2][:4096]).all()
            return "device and host-buffer outputs identical; first 4096 signatures verify with the same challenges"
        def cpu_fn(ns):
            uc, Rc, cc = ref_cpu.sign(s3[:ns], m3[:ns], n3[:ns])
            b = [npv(t) for t in ho]
            assert (uc == b[0][:ns]).all() and (Rc == b[1][:ns]).all() and (cc == b[2][:ns]).all()
            import schnorr_oracle as o
            key = seed_from_u64(0xC3 + rank)  # == o.seed_from_u64 (checked in tests); blocks 0, 1, 777 against the scalar oracle
            assert [int.from_bytes(n3[i].tobytes(), "little") for i in (0, 1, 777)] == [o.nonce_from_block(key, i) for i in (0, 1, 777)]
            return "u, R, c byte-identical to the GPU's; nonces = the oracle's StdRng stream"
        record(name, f"SecretKey::sign, 2^{lg} messages, nonces = from_bytes_wide of consecutive ChaCha12 blocks of StdRng::seed_from_u64 "
                     "(drawn host-side, reduced on the device); outputs u, R (affine), c", m, "signs/s", "sign_batch4",
               lambda: eng.call("sign", m, DEVICE_PTRS, *[P(t) for t in dp], *[P(t) for t in do]),
               lambda: eng.call("sign", m, 0, *[P(t) for t in hp], *[P(t) for t in ho]), m * 96, m * 128, chk, cpu_fn, "sign")
        del hp, dp, ho, do

    if want("c4_verify_vargen_2_22"):
        m = n
        s4, n4, m4 = make_inputs(m, 0xC4 + rank)
        gs = synth_scalars(np.random.RandomState(0x4C4 + rank), m, 27)
        gen = eng.keygen(gs)                       # per-key generator = s * G, as SecretKeyVarGen::random (secret.rs:371-373)
        p4 = eng.keygen_vargen(s4, gen)
        u4, R4, _ = eng.sign_vargen(s4, gen, m4, n4)
        bad4 = corrupt_mask(m)
        mode = np.arange(m) % 4
        u4[bad4 & (mode == 0), 0] ^= 1
        m4[bad4 & (mode == 1), 0] ^= 1
        sel = bad4 & (mode == 2); p4[sel] = np.roll(p4, -1, axis=0)[sel]
        sel = bad4 & (mode == 3); gen[sel] = np.roll(gen, -1, axis=0)[sel]
        arrs = (p4, gen, u4, R4, m4)
        hp = [pinned(a) for a in arrs]
        dp = [t.to(dev) for t in hp]
        hb, db = torch.zeros(m // 32, dtype=torch.int32).pin_memory(), torch.zeros(m // 32, dtype=torch.int32, device=dev)
        def chk():
            assert (unpack(db, m) == ~bad4).all() and (unpack(npv(hb), m) == ~bad4).all()
            return "verdict == not corrupted for all tuples (10 % corrupted: u, message, pk, generator)"
        def cpu_fn(ns):
            okc, _ = ref_cpu.verify_vargen(*[a[:ns] for a in arrs])
            assert (okc == ~bad4[:ns]).all()
            return "verdicts identical to the GPU's"
        record("c4_verify_vargen_2_22", f"PublicKeyVarGen::verify, 2^{args.log2_batch} tuples, per-key generators, 10% corrupted in four ways",
               m, UNIT, "verify_vargen_affine", lambda: eng.call("verify_vargen", m, fl, *[P(t) for t in dp], P(db), None),
               lambda: eng.call("verify_vargen", m, POINTS_AFFINE, *[P(t) for t in hp], P(hb), None), m * 256, m // 8, chk, cpu_fn,
               "verify_vargen_affine")
        del hp, dp

    if want("verify_bytes_2_20"):
        m = min(n, 1 << 20)
        pkb = eng.points_compress(pk[:m])
        sigb = np.concatenate([u[:m].view(np.uint8).reshape(m, 32), eng.points_compress(R[:m])], axis=1)
        msgb = eng.fq_from_mont(msg[:m]).view(np.uint8).reshape(m, 32)
        hp = [pinned(np.ascontiguousarray(a)) for a in (pkb, sigb, msgb)]
        dp = [t.to(dev) for t in hp]
        hb, db = torch.zeros(m // 32, dtype=torch.int32).pin_memory(), torch.zeros(m // 32, dtype=torch.int32, device=dev)
        hi, di = torch.zeros(m // 32, dtype=torch.int32).pin_memory(), torch.zeros(m // 32, dtype=torch.int32, device=dev)
        def chk():
            assert (unpack(db, m) == ~bad[:m]).all() and (unpack(npv(hb), m) == ~bad[:m]).all()
            assert not unpack(di, m).any() and not unpack(npv(hi), m).any()
            return "verdicts equal those of the limb-level call on the same tuples; no tuple invalid"
        record("verify_bytes_2_20", "PublicKey::from_bytes(pk)?.verify(&Signature::from_bytes(sig)?, BlsScalar::from_bytes(msg)?): 32 + 64 + 32 wire "
               "bytes per tuple, decompression on the device, 10% corrupted", m, UNIT, "verify_bytes",
               lambda: eng.call("verify_bytes", m, DEVICE_PTRS, *[P(t) for t in dp], P(db), P(di)),
               lambda: eng.call("verify_bytes", m, 0, *[P(t) for t in hp], P(hb), P(hi)), m * 128, m // 4, chk)
        del hp, dp

    # ---- the typed host API with pageable memory (C++ mirror of the reference's types) -------------------------------
    typed = None
    exe = os.path.join(ROOT, "build", "bench_typed")
    if not args.no_extras and not only and rank == 0 and world == 1 and os.path.exists(exe):
        try:
            out = subprocess.run([exe, "20", "2"], capture_output=True, text=True, timeout=300,
                                 env=dict(os.environ, CUDA_VISIBLE_DEVICES=os.environ.get("CUDA_VISIBLE_DEVICES", str(local))))
            typed = json.loads(out.stdout) if out.returncode == 0 else {"error": out.stderr[-300:]}
        except Exception as ex:  # pragma: no cover
            typed = {"error": repr(ex)}

    # ---- strong scaling: ONE context over all N devices, one 2^22 batch in host buffers ------------------------------
    strong = None
    if world > 1 and not args.no_extras and not only:
        barrier()
        # the other ranks wait on the HOST (TCP store), not in an NCCL barrier: a pending NCCL collective is a kernel spinning on
        # their GPUs, which are exactly the devices rank 0's multi-device context is about to measure
        store = dist.distributed_c10d._get_default_store()
        if rank != 0:
            store.wait(["sb200_strong_done"])
        if rank == 0:
            try:
                big = Engine(list(range(world)))
                call = lambda: big.call("verify", n, POINTS_AFFINE, P(h_pk), P(h_u), P(h_R), P(h_msg), P(h_bm), None)
                call(); call()
                t0 = time.perf_counter()
                for _ in range(ksteps):
                    call()
                dt = (time.perf_counter() - t0) / ksteps
                assert (unpack(npv(h_bm), n) == ~bad).all()
                per_gpu_ms = ms_step / world
                strong = {"workload": f"one sb200 context over {world} devices, ONE batch of 2^{args.log2_batch} tuples in pinned host buffers, "
                                      "one host thread per device, no collective", "n_total": n, "value": n / dt, "unit": UNIT, "ms_per_step": dt * 1e3,
                          "ideal_ms_if_compute_only": per_gpu_ms, "h2d_bytes_per_step": h2d,
                          "h2d_gbs_implied": h2d / dt / 1e9,
                          "limiter": "compute" if dt * 1e3 < 1.3 * per_gpu_ms else "host-to-device copies / launch latency of the per-device pipeline"}
                big.close()
            except Exception as ex:  # pragma: no cover
                strong = {"error": repr(ex)}
            store.set("sb200_strong_done", "1")
        barrier()

    if rank == 0:
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32",
            "data": "synthetic",
            "config": {"workload": f"single-key PublicKey::verify, batch 2^{args.log2_batch} per GPU, 10% corrupted signatures, "
                                   "affine (u,v) Montgomery inputs; sharded by tuple index, no collective",
                       "batch_per_gpu": n, "l2": "inputs (1 GiB) larger than L2; no flush needed",
                       "round_constants": os.environ.get("SB200_ARK") or "cumsum"},
            "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "timing": "wall clock around the blocking host-buffer call (pinned host memory, chunked 2-stream pipeline)"},
            "gpu_launches": launches,
            "clocks": sampler.result(),
            "roofline": roof,
            "cpu_baseline": cpu,
            "configs": configs,
            "e2e_typed": typed,
            "strong_scaling": strong,
        }
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    eng.close()


if __name__ == "__main__":
    main()
