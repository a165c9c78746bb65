#!/usr/bin/env python3
"""Headline benchmark: BLS12-381 G1 MSM points/sec at 2^20 scalars (BASELINE.json `metric`).

    python bench.py --gpus N --steps K --warmup W            # our CUDA path (default N=1)
    python bench.py --impl reference --steps K --warmup W    # the reference algorithm on host cores

One "step" = one complete MSM (curve.ts:863-905 `pippenger` semantics) over one batch of synthetic
(point, scalar) terms:  points P_i = k_i*G, scalars uniform in [0, n).  SURVEY §8(d): points/s = N / wall time of ONE
MSM, so the timed region runs the K steps one after the other (each call returns the affine result before the next
starts); the throughput with several MSMs in flight is a named companion (`pipelined`), not the headline.
At N GPUs (default "scaling": "strong" = the metric's configuration: 2^20 terms IN TOTAL) the term array is sharded
across the ranks and one step is one nmsm_msm_sharded call: every rank accumulates its shard into the full bucket array,
window w's buckets go to rank w % N (NCCL send/recv inside the library), the owner folds + reduces its windows, one small
all-gather + fold finishes (nmsm/dist.py).  `--scaling weak` (2^logn terms PER GPU, one MSM of N*2^logn terms) is kept
as a companion mode.

Timed numbers:
  value  — whole-job points/s with inputs already resident in HBM (nmsm_msm_device / nmsm_msm_sharded), serial steps
  e2e    — same metric through the host-buffer entry points (pinned host inputs, H2D inside), serial steps
  roofline — modmul-bound integer roofline of the dominant kernel (k_accumulate): executed field
             multiplications / CUDA-event time, against the register-resident Montgomery-multiply
             microbenchmark measured in the same run; HBM figures alongside
  cpu_baseline — the reference algorithm restated for the CPU (oracle/), timed on a bounded sample
"""
import argparse
import ctypes
import json
import os
import random
import subprocess
import sys
import threading
import time

os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")  # before any CUDA context exists (see nmsm/_lib.py)
os.environ.setdefault("NCCL_MIN_P2P_NCHANNELS", "16")       # before any NCCL communicator exists (see nmsm/_lib.py)
os.environ.setdefault("NCCL_MAX_P2P_NCHANNELS", "32")
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "noble-curves_b200"))
sys.path.insert(0, ROOT)

BLS_G1 = 4
POINT_BYTES = 96
BLS_N = 0x73EDA753299D7D483339D80809A1D80553BDA402FFFE5BFEFFFFFFFF00000001
BLS_GX = 0x17F1D3A73197D7942695638C4FA9AC0FC3688C4F9774B905A14E3A3F171BAC586C55E83FF97A1AEFFB3AF00ADB22C6BB
BLS_GY = 0x08B3F481E3AAA0F1A09E30ED741D8AE4FCF5E095D5D00AF600DB18CB2C04B3EDD03CC744A2888AE40CAA232946C5E7E1


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--logn", type=int, default=20, help="log2 of the MSM size (headline: 20)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-fixed-base", action="store_true", help="skip the fixed-base table and any-point companion measurements")
    ap.add_argument("--no-pipelined", action="store_true", help="skip the MSMs-in-flight companion measurement")
    ap.add_argument("--window", type=int, default=0, help="force window bits c (0 = cost model)")
    ap.add_argument("--in-flight", type=int, default=4, choices=[2, 3, 4], help="MSMs kept in flight in the `pipelined` companion")
    ap.add_argument("--scaling", default="strong", choices=["weak", "strong"],
                    help="N>1: strong (default, the metric's config) = 2^logn terms in total; weak = 2^logn terms PER GPU")
    ap.add_argument("--groups", type=int, default=0, help="force the window-group count of the pipeline (0 = automatic)")
    ap.add_argument("--configs", action="store_true",
                    help="instead of the headline line: time every BASELINE.json config on one GPU (one JSON line, key `configs`)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the result of the last timed step as DIR/<name>.npy (float64), to compare two builds output for "
                         "output; the inputs depend only on the arguments")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.configs):
        ap.error("--dump-outputs applies to the headline GPU run (not --impl reference or --configs)")
    return args


def dump_outputs(dirname, xy: bytes, is_inf: int):
    """What nmsm_msm_device hands its caller for one BLS12-381 G1 MSM: the affine result (x, y), each 48 bytes little-endian,
    stored as 12 little-endian 32-bit limbs per coordinate (exact in float64), and the point-at-infinity flag."""
    import numpy as np

    os.makedirs(dirname, exist_ok=True)
    limbs = np.frombuffer(xy, dtype="<u4").reshape(2, POINT_BYTES // 8)
    np.save(os.path.join(dirname, "msm_affine_xy_limbs.npy"), limbs.astype(np.float64))
    np.save(os.path.join(dirname, "msm_is_infinity.npy"), np.array([is_inf], dtype=np.float64))


# --------------------------------------------------------------------------------------------
# clocks sampler (B200_PROFILING.md "clocks DURING the timed region")
# --------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "20"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# --------------------------------------------------------------------------------------------
# synthetic inputs
# --------------------------------------------------------------------------------------------
def make_terms(nmsm, n, seed):
    """n random (point, scalar) terms; points are generated ON THE GPU as k_i*G (nmsm_mul_batch).
    Returns (points bytes, scalars bytes, expected total scalar sum k_i*s_i mod n)."""
    rnd = random.Random(seed)
    ks = [rnd.randrange(1, BLS_N) for _ in range(n)]
    sc = [rnd.randrange(BLS_N) for _ in range(n)]
    g = BLS_GX.to_bytes(48, "little") + BLS_GY.to_bytes(48, "little")
    pts, infs = nmsm.mul_batch_packed(BLS_G1, g * n, b"".join(k.to_bytes(32, "little") for k in ks), n, False)
    total = sum(k * s for k, s in zip(ks, sc)) % BLS_N
    return pts, b"".join(s.to_bytes(32, "little") for s in sc), total


def expected_point(nmsm, total):
    """(sum k_i s_i)*G computed by the GPU scalar-mult path (itself parity-tested against the oracle)."""
    if total == 0:
        return bytes(96), 1
    g = BLS_GX.to_bytes(48, "little") + BLS_GY.to_bytes(48, "little")
    out, infs = nmsm.mul_batch_packed(BLS_G1, g, total.to_bytes(32, "little"), 1, True)
    return out, infs[0]


# --------------------------------------------------------------------------------------------
# reference arm: the reference's algorithm on host cores (oracle/ is allowed here only)
# --------------------------------------------------------------------------------------------
def cpu_reference(n_sample, seed, max_seconds=30.0):
    """Times the CPU restatement of noble's pippenger (same window rule, unsigned windows, complete
    RCB additions) on a bounded sample.  Prefers the C port (oracle/ref_msm.c, all host threads);
    falls back to the Python-int oracle on a smaller sample."""
    from oracle import cpu_baseline

    return cpu_baseline.time_bls_g1_msm(n_sample, seed, max_seconds)


def run_reference(args, real_stdout):
    """`--impl reference`: the reference's algorithm on this box's host cores (rank 0 only under torchrun).
    Inputs are generated once; each step is one timed run of the C port on the same workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import cpu_baseline as CB

    n_full = 1 << args.logn
    n_sample = CB.choose_sample(30.0, args.logn)
    w = CB.Workload(n_sample, 1)
    times = [w.run() for _ in range(args.warmup + args.steps)][args.warmup:]
    res = CB.describe(n_sample, sum(times) / len(times), args.logn)
    pts_per_s = res["points_per_s_at_full_size"]
    line = {
        "impl": "reference",
        "metric": "BLS12-381 G1 MSM points/sec at 2^%d scalars" % args.logn,
        "value": pts_per_s, "unit": "points/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * n_full / pts_per_s, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "u64-limb integer (381-bit Fp, Montgomery)", "data": "synthetic",
        "config": {"workload": "BLS12-381 G1 MSM, 2^%d terms, reference algorithm (curve.ts:863-905) on host cores; "
                               "host-only: the same single-box workload at every --gpus" % args.logn},
        "cpu_baseline": {"value": pts_per_s, "unit": "points/s", "cores": res["cores"], "kind": res["kind"],
                         "sample": res["sample"]},
        "e2e": {"value": pts_per_s, "unit": "points/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    _emit(real_stdout, line)


# --------------------------------------------------------------------------------------------
# our arm
# --------------------------------------------------------------------------------------------
def _claim_stdout():
    """stdout must carry exactly ONE JSON line, but native libraries write there too (NCCL prints its version banner
    to fd 1 when the launch environment sets NCCL_DEBUG=VERSION/WARN).  Point fd 1 at stderr for the whole run and keep
    the real stdout for the final line."""
    sys.stdout.flush()
    real = os.dup(1)
    os.dup2(2, 1)
    return real


def _emit(real_stdout_fd, line: dict):
    sys.stdout.flush()
    os.write(real_stdout_fd, (json.dumps(line) + "\n").encode())


# --------------------------------------------------------------------------------------------
# the five BASELINE.json configs on one GPU (companion table; the parity tests of the same configs are in tests/)
# --------------------------------------------------------------------------------------------
def run_configs(args, real_stdout):
    """Each config is timed through the host-buffer C-ABI entry point a caller of the reference would use (H2D inside) and,
    for the MSMs, also as device time of the pipeline (library events).  Results are checked on the GPU itself by the
    scalar-in-the-exponent identity  sum s_i * (k_i G) = (sum k_i s_i) G  (test/slow-curves.test.ts:204-233); the bit-exact
    comparison against the oracle for these very configs is tests/test_gpu_parity.py::test_config_*."""
    import nmsm

    nmsm.init(0)
    rows = []

    def best_of(fn, reps):
        best = 1e9
        for _ in range(reps):
            t0 = time.perf_counter()
            fn()
            best = min(best, time.perf_counter() - t0)
        return best

    def pack(v, nbytes):
        return v.to_bytes(nbytes, "little") if isinstance(v, int) else b"".join(c.to_bytes(nbytes, "little") for c in v)

    def msm_row(idx, C, logn, seed):
        n = 1 << logn
        order, cid, fb = C.Fn.ORDER, C.CURVE_ID, C.FP_BYTES
        rnd = random.Random(seed)
        ks = [rnd.randrange(1, order) for _ in range(n)]
        sc = [rnd.randrange(order) for _ in range(n)]
        g = pack(C.BASE.x, fb) + pack(C.BASE.y, fb)
        scb = b"".join(s_.to_bytes(32, "little") for s_ in sc)
        pts, _ = nmsm.mul_batch_packed(cid, g * n, b"".join(k.to_bytes(32, "little") for k in ks), n, False)
        total = sum(k * s_ for k, s_ in zip(ks, sc)) % order
        exp, _ = nmsm.mul_batch_packed(cid, g, total.to_bytes(32, "little"), 1, True)
        res = {}

        def run():
            res["o"] = nmsm.msm_packed(cid, pts, scb, n)

        run()
        run()
        best = best_of(run, args.steps if args.steps < 8 else 8)
        ms, info = nmsm.last_timing()
        rows.append({"config": idx, "what": "%s Pippenger MSM, 2^%d random terms" % (C.NAME, logn), "n": n,
                     "ms_host_buffers": best * 1e3, "ms_device": ms["total"], "points_per_s_device": n / (ms["total"] * 1e-3),
                     "plan": {"c": info.c, "windows": info.windows, "sorted_entries": info.sorted_entries},
                     "check": "ok: equals (sum k_i s_i)*G" if res["o"][0] == exp and res["o"][1] == 0 else "MISMATCH"})

    # config 0: secp256k1 Point.multiply batch of 1024 random scalars (benchmark/point.ts shape: one public key, many scalars)
    C = nmsm.CURVES["secp256k1"]
    order = C.Fn.ORDER
    rnd = random.Random(11)
    b0 = rnd.randrange(1, order)
    g = pack(C.BASE.x, 32) + pack(C.BASE.y, 32)
    pk, _ = nmsm.mul_batch_packed(0, g, b0.to_bytes(32, "little"), 1, False)
    ks = [rnd.randrange(1, order) for _ in range(1024)]
    ksb = b"".join(k.to_bytes(32, "little") for k in ks)
    res = {}

    def run0():
        res["o"] = nmsm.mul_batch_packed(0, pk * 1024, ksb, 1024, False)

    run0()
    best = best_of(run0, 5)
    exp, _ = nmsm.mul_batch_packed(0, g * 1024, b"".join(((k * b0) % order).to_bytes(32, "little") for k in ks), 1024, False)
    rows.append({"config": 0, "what": "secp256k1 Point.multiply, batch of 1024 random scalars", "n": 1024, "ms_host_buffers": best * 1e3,
                 "multiplies_per_s": 1024 / best, "check": "ok: k_i*(b*G) == (k_i*b)*G" if res["o"][0] == exp else "MISMATCH"})
    msm_row(1, nmsm.CURVES["bls12_381_G1"], 16, 101)
    msm_row(2, nmsm.CURVES["bn254_G1"], 20, 102)
    msm_row(3, nmsm.CURVES["bls12_381_G2"], 18, 103)
    # config 4: ed25519 batch verification of 2^16 signatures (1024 fresh signatures tiled x64)
    try:
        from cryptography.hazmat.primitives import serialization
        from cryptography.hazmat.primitives.asymmetric.ed25519 import Ed25519PrivateKey

        base = []
        for i in range(1024):
            sk = Ed25519PrivateKey.generate()
            msg = (b"noble-curves_b200 bench %d" % i) * (1 + i % 3)
            base.append((sk.sign(msg), msg, sk.public_key().public_bytes(serialization.Encoding.Raw, serialization.PublicFormat.Raw)))
        reps = (1 << 16) // len(base)
        sigs, msgs, pks = [b[0] for b in base] * reps, [b[1] for b in base] * reps, [b[2] for b in base] * reps
        z = os.urandom(16 * len(sigs))

        def run4():
            res["v"] = nmsm.ed25519_verify_batch(sigs, msgs, pks, z)

        run4()
        best = best_of(run4, 3)
        # the C-ABI call alone, arrays packed once outside the timed region (what a native caller pays)
        import struct

        offs = [0]
        for m in msgs:
            offs.append(offs[-1] + len(m))
        packed = (b"".join(sigs), b"".join(pks), b"".join(msgs), struct.pack("<%dQ" % (len(sigs) + 1), *offs), len(sigs), z)

        def run4p():
            res["p"] = nmsm.ed25519_verify_batch_packed(*packed)

        run4p()
        best_p = best_of(run4p, 5)
        bad = list(sigs)
        bad[777] = bad[777][:40] + bytes([bad[777][40] ^ 1]) + bad[777][41:]
        rej = nmsm.ed25519_verify_batch(bad, msgs, pks, z)
        rows.append({"config": 4, "what": "ed25519 batch verification, 2^16 signatures (Edwards MSM of 2^17 + 1 terms)", "n": len(sigs),
                     "ms_host_buffers": best_p * 1e3, "signatures_per_s": len(sigs) / best_p,
                     "ms_through_python_binding": best * 1e3,
                     "check": "ok: valid batch accepted, one corrupted signature rejected"
                     if res["v"] == (True, -1) and res["p"] == (True, -1) and not rej[0] else "MISMATCH"})
    except ImportError as e:
        rows.append({"config": 4, "what": "ed25519 batch verification", "skipped": "no signer available: %r" % (e,)})
    _emit(real_stdout, {"configs": rows, "n_gpus": 1, "data": "synthetic",
                        "note": "companion table of bench.py --configs; the headline metric is the default bench.py line"})


def main():
    args = parse_args()
    real_stdout = _claim_stdout()
    if args.impl == "reference":
        run_reference(args, real_stdout)
        return
    if args.configs:
        run_configs(args, real_stdout)
        return

    import torch
    import torch.distributed as dist

    import nmsm
    from nmsm import dist as nd

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the MSM path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    nmsm.init(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        nd.init()
    lib = nmsm._lib.load()
    if args.window:
        nmsm.set_window_bits(args.window)
    if args.groups:
        nmsm.set_window_groups(args.groups)

    # strong (default): the 2^logn terms of ONE MSM are split across the GPUs; weak: 2^logn terms per GPU
    scaling = args.scaling if world > 1 else "strong"
    n_total = (1 << args.logn) * (world if scaling == "weak" else 1)
    lo, hi = nd.shard_bounds(n_total, world, rank)
    n_local = hi - lo
    # every rank generates only its own shard; seeds make shards disjoint and reproducible
    pts_b, sc_b, total_local = make_terms(nmsm, n_local, 1000 + rank)
    d_pts = torch.frombuffer(bytearray(pts_b), dtype=torch.uint8).to(dev)
    d_sc = torch.frombuffer(bytearray(sc_b), dtype=torch.uint8).to(dev)
    out = ctypes.create_string_buffer(POINT_BYTES)
    inf = ctypes.c_int(0)
    vp = lambda b: ctypes.cast(b, ctypes.c_void_p)  # noqa: E731

    if world > 1:
        totals = [None] * world
        dist.all_gather_object(totals, total_local)
        total = sum(totals) % BLS_N
    else:
        total = total_local
    exp_xy, exp_inf = expected_point(nmsm, total)

    def check_result(o=out, f=inf):
        assert o.raw == exp_xy and f.value == exp_inf, "MSM result does not match (sum k_i s_i)*G"

    def step_device():  # ONE complete MSM, inputs resident in HBM
        if world == 1:
            nmsm._lib.check(lib.nmsm_msm_device(BLS_G1, d_pts.data_ptr(), d_sc.data_ptr(), n_local, vp(out), ctypes.byref(inf)))
        else:
            nmsm._lib.check(lib.nmsm_msm_sharded(BLS_G1, d_pts.data_ptr(), d_sc.data_ptr(), n_local, n_total, lo, 1, vp(out),
                                                 ctypes.byref(inf)))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    W = max(args.warmup, 3)
    # ---- (1) profiling pass (single GPU): linear pipeline, per-kernel CUDA-event times, executed-addition counts ----
    kern_ms, acc_ms, lin_ms, prof_info = {}, [], [], None
    if world == 1:
        nmsm.set_profiling(True)
        for _ in range(W):
            step_device()
        check_result()
        for _ in range(args.steps):
            step_device()
            ms, prof_info = nmsm.last_timing()
            acc_ms.append(ms["accumulate"])
            lin_ms.append(ms["total"])
            for k, v in ms.items():
                kern_ms[k] = kern_ms.get(k, 0.0) + v / args.steps
        nmsm.set_profiling(False)

    # ---- (2) THE TIMED REGION: K serial steps, one complete MSM each (SURVEY §8d: N / wall time of one MSM) -----------
    # clocks are sampled (nvidia-smi, 20 ms period) from the warm-up of the device-resident timed region to the end of the
    # end-to-end timed region: the two regions are a few hundred ms in total, shorter than nvidia-smi's start-up alone
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.5)
    for _ in range(W):
        step_device()
    check_result()
    dev_ms = []
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_device()
        dev_ms.append(nmsm.last_timing()[0]["total"])
    barrier()
    elapsed = max_over_ranks(time.perf_counter() - t0)
    check_result()
    last_xy, last_inf = out.raw, inf.value  # `out` is reused by the companion measurements below
    main_info = nmsm.last_timing()[1]
    device_ms = max_over_ranks(sum(dev_ms) / len(dev_ms))
    value = n_total * args.steps / elapsed

    # ---- (3) end to end: the same serial steps through the host-buffer entry points (pinned inputs, H2D inside) -------
    h_pts = lib.nmsm_host_alloc(max(16, len(pts_b)))
    h_sc = lib.nmsm_host_alloc(max(16, len(sc_b)))
    ctypes.memmove(h_pts, pts_b, len(pts_b))
    ctypes.memmove(h_sc, sc_b, len(sc_b))

    def step_e2e():
        if world == 1:
            nmsm._lib.check(lib.nmsm_msm(BLS_G1, h_pts, h_sc, n_local, vp(out), ctypes.byref(inf)))
        else:
            nmsm._lib.check(lib.nmsm_msm_sharded(BLS_G1, h_pts, h_sc, n_local, n_total, lo, 0, vp(out), ctypes.byref(inf)))

    for _ in range(W):
        step_e2e()
    check_result()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_e2e()
    barrier()
    e2e_elapsed = max_over_ranks(time.perf_counter() - t0)
    clocks = sampler.stop() if rank == 0 else None
    check_result()
    e2e_value = n_total * args.steps / e2e_elapsed

    # ---- (4) companion: several MSMs in flight (nmsm_msm_submit / collect over the slots) ----------------------------
    NF = args.in_flight
    pipelined = None

    def run_pipelined(steps, submit):
        outs = [ctypes.create_string_buffer(POINT_BYTES) for _ in range(NF)]
        infs = [ctypes.c_int(0) for _ in range(NF)]

        def take(s):
            nmsm._lib.check(lib.nmsm_msm_collect(s, vp(outs[s]), ctypes.byref(infs[s])))
            check_result(outs[s], infs[s])

        for i in range(steps):
            s = i % NF
            if i >= NF:  # the slot still holds step i - NF
                take(s)
            submit(s)
        for j in range(max(0, steps - NF), steps):
            take(j % NF)

    def submit_device(slot):
        if world == 1:
            nmsm._lib.check(lib.nmsm_msm_submit(BLS_G1, d_pts.data_ptr(), d_sc.data_ptr(), n_local, 1, slot))
        else:
            nmsm._lib.check(lib.nmsm_msm_sharded_submit(BLS_G1, d_pts.data_ptr(), d_sc.data_ptr(), n_local, n_total, lo, 1, slot))

    def submit_host(slot):
        if world == 1:
            nmsm._lib.check(lib.nmsm_msm_submit(BLS_G1, h_pts, h_sc, n_local, 0, slot))
        else:
            nmsm._lib.check(lib.nmsm_msm_sharded_submit(BLS_G1, h_pts, h_sc, n_local, n_total, lo, 0, slot))

    if not args.no_pipelined:
        pipelined = {"in_flight": NF}
        for key, submit in (("device", submit_device), ("e2e", submit_host)):
            run_pipelined(2 * NF + 1, submit)  # touches every slot (workspace allocation) before the timed loop
            barrier()
            t0 = time.perf_counter()
            run_pipelined(args.steps, submit)
            barrier()
            el = max_over_ranks(time.perf_counter() - t0)
            pipelined[key] = {"value": n_total * args.steps / el, "unit": "points/s", "ms_per_step": 1e3 * el / args.steps}
        pipelined["note"] = ("companion, NOT the headline: the same K MSMs with several kept in flight on separate slots "
                             "(nmsm_msm_submit / nmsm_msm_collect); throughput of a prover that has independent MSMs to run")
    lib.nmsm_host_free(h_pts)
    lib.nmsm_host_free(h_sc)

    # ---- companion: the same MSM over a device-resident point set with a fixed-base table (SURVEY §8 f4) -------------
    fixed = None
    if world == 1 and not args.no_fixed_base:
        h, tc, lv = ctypes.c_uint64(0), ctypes.c_int(0), ctypes.c_int(0)
        nmsm._lib.check(lib.nmsm_points_upload(BLS_G1, ctypes.cast(ctypes.c_char_p(pts_b), ctypes.c_void_p), n_local, ctypes.byref(h)))
        t0 = time.perf_counter()
        nmsm._lib.check(lib.nmsm_points_precompute(h, 0, ctypes.byref(tc), ctypes.byref(lv)))
        t_pre = time.perf_counter() - t0

        def step_fixed():
            nmsm._lib.check(lib.nmsm_msm_points_submit(h, d_sc.data_ptr(), n_local, 1, 0))
            nmsm._lib.check(lib.nmsm_msm_collect(0, vp(out), ctypes.byref(inf)))

        nmsm.set_profiling(True)
        for _ in range(3):
            step_fixed()
        check_result()
        fms, finfo = nmsm.last_timing()
        nmsm.set_profiling(False)
        for _ in range(3):
            step_fixed()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            step_fixed()
        barrier()
        f_el = time.perf_counter() - t0
        check_result()
        fixed = {"value": n_local * args.steps / f_el, "unit": "points/s", "ms_per_step": 1e3 * f_el / args.steps,
                 "table": {"window_bits": tc.value, "levels": lv.value, "bytes": lv.value * 2 * n_local * 96,
                           "precompute_ms": t_pre * 1e3},
                 "plan": {"c": finfo.c, "windows": finfo.windows, "sorted_entries": finfo.sorted_entries},
                 "kernel_ms_breakdown_linear": {k: round(v, 4) for k, v in fms.items()},
                 "note": "device-resident point set + table 2^(c*j)*P (nmsm_points_precompute), serial steps; companion to "
                         "`value`, which stays the general MSM with points passed per call"}
        lib.nmsm_points_free(h)

    # ---- companion: the same MSM under NMSM_BLS12_381_G1_ANY (what nmsm.pippenger selects for unvalidated points) -----
    any_point = None
    if world == 1 and not args.no_fixed_base:
        ANY = 6
        for _ in range(3):
            nmsm._lib.check(lib.nmsm_msm_device(ANY, d_pts.data_ptr(), d_sc.data_ptr(), n_local, vp(out), ctypes.byref(inf)))
        check_result()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            nmsm._lib.check(lib.nmsm_msm_device(ANY, d_pts.data_ptr(), d_sc.data_ptr(), n_local, vp(out), ctypes.byref(inf)))
        torch.cuda.synchronize()
        a_el = (time.perf_counter() - t0) / args.steps
        any_point = {"value": n_local / a_el, "unit": "points/s", "ms_per_step": 1e3 * a_el,
                     "note": "curve id NMSM_BLS12_381_G1_ANY (no endomorphism, 16 windows): valid for EVERY on-curve point; "
                             "the host mirror's pippenger picks it unless all inputs are known subgroup members (the bench "
                             "points k_i*G are, so the headline uses id 4); serial steps"}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline ---------------------------------------------------------------------------------------------------
    peak = 0.0
    for (bps, thr, ilp) in ((4, 128, 1), (8, 128, 1), (4, 256, 1), (4, 128, 2), (8, 128, 2), (2, 256, 2)):
        peak = max(peak, nmsm.bench_modmul(1, bps, thr, 3000, ilp))
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    info = prof_info if prof_info is not None else main_info
    roofline = {"bound": "int-modmul", "kernel": "k_accumulate<BLS12-381 G1>", "unit": "Gmodmul/s (381-bit Montgomery)",
                "peak": peak / 1e9,
                "peak_source": "nmsm_bench_modmul: register-resident dependent mont_mul<FpBls381> chains on all SMs, same run",
                "plan": {"c": info.c, "windows": info.windows, "buckets_per_window": info.buckets_per_window,
                         "entries_per_thread": info.entries_per_thread, "sorted_entries": info.sorted_entries,
                         "window_groups_timed_region": main_info.window_groups}}
    if world == 1:
        acc_t = sum(acc_ms) / len(acc_ms) * 1e-3
        # executed field multiplications of k_accumulate.  Every sorted entry except those that START an accumulator (a copy)
        # ends in one mixed addition, madd-2008-s 8M + 2S = 10; a same-bucket pair is first added in affine (3 for its share
        # of the warp's batch inversion + 2M + 1S) and then takes ONE mixed addition: 16 for two entries instead of 20, i.e.
        # -4 per pair; every thread pays 12 for the prefix / suffix products of the warp-shared inversion.
        madds = info.sorted_entries - info.bucket_starts - info.bucket_pairs
        madd_modmuls = 10 * (info.sorted_entries - info.bucket_starts) - 4 * info.bucket_pairs + \
            (12 * info.accumulate_threads if info.bucket_pairs else 0)  # the warp scan only exists in the paired build
        achieved = madd_modmuls / acc_t
        # whole MSM, executed: mixed additions + bucket reduction (2 additions per bucket of 12M+2S) + Horner doublings (6M+3S)
        W_, B_ = info.windows, info.buckets_per_window
        whole_modmuls = madd_modmuls + W_ * 2 * B_ * 14 + (W_ - 1) * info.c * 9
        # algorithmic bytes of k_accumulate per launch: per sorted entry one 96-byte gathered affine point + its 4-byte index;
        # per accumulator start one 192-byte XYZZ accumulator written (buckets, heads, tails)
        acc_bytes_alg = info.sorted_entries * (96 + 4) + info.bucket_starts * 192
        one_ms = 1e3 * elapsed / args.steps
        roofline.update({
            "achieved": achieved / 1e9, "frac": achieved / peak if peak > 0 else None,
            "mixed_additions_executed": madds, "affine_pair_additions_executed": info.bucket_pairs,
            "accumulator_starts": info.bucket_starts, "accumulate_threads": info.accumulate_threads,
            "modmul_per_launch": madd_modmuls, "kernel_ms": acc_t * 1e3,
            "whole_msm": {"modmul_executed": whole_modmuls, "ms": one_ms,
                          "frac": (whole_modmuls / (one_ms * 1e-3)) / peak if peak > 0 else None,
                          "ms_linear_pipeline": sum(lin_ms) / len(lin_ms),
                          "note": "executed field multiplications of one MSM / wall time of one serial step / peak"},
            "hbm": {"achieved_gbs": acc_bytes_alg / acc_t / 1e9, "peak_gbs": hbm_peak,
                    "frac": acc_bytes_alg / acc_t / 1e9 / hbm_peak, "algorithmic_bytes": acc_bytes_alg,
                    "peak_source": "MEASURED_PEAKS.json" if peaks else "fallback 6.65 TB/s"},
            "traffic": None,
            "kernel_ms_breakdown_linear": {k: round(v, 4) for k, v in kern_ms.items()},
        })
        traffic_file = os.path.join(ROOT, "profiles", "traffic_k_accumulate.json")
        if os.path.exists(traffic_file):
            try:
                roofline["traffic"] = json.load(open(traffic_file)).get("dram_bytes_per_launch")
            except Exception:
                pass
    else:
        roofline.update({"achieved": None, "frac": None, "traffic": None,
                         "note": "per-kernel profile is taken at N=1 (profiling forces the linear pipeline); at N>1 see device_ms_per_step"})

    cpu = None
    if not args.no_cpu_baseline and world == 1:
        try:
            r = cpu_reference(None, 1)
            cpu = {"value": r["points_per_s_at_full_size"], "unit": "points/s", "cores": r["cores"], "kind": r["kind"],
                   "sample": r["sample"]}
        except Exception as e:  # never lose the GPU line because the CPU leg failed
            cpu = {"value": None, "unit": "points/s", "cores": 0, "kind": "port", "sample": "failed: %r" % (e,)}

    nccl_ver = None
    if world > 1:
        v = ctypes.c_int(0)
        lib.nmsm_dist_info(None, None, ctypes.byref(v))
        nccl_ver = v.value
    line = {
        "metric": "BLS12-381 G1 MSM points/sec at 2^%d scalars" % args.logn,
        "value": value, "unit": "points/s", "n_gpus": world, "steps": args.steps, "warmup": W,
        "ms_per_step": 1e3 * elapsed / args.steps, "device_ms_per_step": device_ms,
        "higher_is_better": True, "scaling": scaling,
        "vs_baseline": None, "dtype": "u32-limb integer (381-bit Fp, Montgomery)", "data": "synthetic",
        "config": {"workload": ("BLS12-381 G1 Pippenger MSM, 2^%d random terms (points k_i*G, uniform scalars) IN TOTAL" % args.logn)
                   if scaling == "strong" else
                   ("BLS12-381 G1 Pippenger MSM, 2^%d terms per GPU: one MSM of %d*2^%d terms" % (args.logn, world, args.logn)),
                   "terms": n_total, "terms_per_gpu": n_local,
                   "parallelism": "1 GPU" if world == 1 else
                   ("term-sharded x%d; per-window bucket exchange to the window owner w %% N inside the library (%s), owner "
                    "fold + reduce, ncclAllGather of %d-byte weighted window sums"
                    % (world, "owners read the peers' buckets in place over NVLink peer memory, fused into the fold kernel"
                       if lib.nmsm_dist_exchange_mode() == 2 else "grouped ncclSend / ncclRecv on the library's own stream", 192)),
                   "steps_are": "serial: one complete MSM per step, result on the host before the next step starts",
                   "l2": "inputs + workspace (>= 450 MB at 2^20 terms) exceed the 126 MB L2; no flush needed",
                   "nccl_version": nccl_ver},
        "e2e": {"value": e2e_value, "unit": "points/s", "ms_per_step": 1e3 * e2e_elapsed / args.steps,
                "h2d_bytes_per_step": len(pts_b) + len(sc_b), "d2h_bytes_per_step": POINT_BYTES + 24, "steps": args.steps},
        "gpu_launches": main_info.launches * args.steps * world,  # our kernels inside the timed region (every rank runs its own)
        "clocks": clocks,
        "roofline": roofline,
        "cpu_baseline": cpu,
        "pipelined": pipelined,
        "fixed_base": fixed,
        "any_point": any_point,
    }
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, last_xy, last_inf)
    _emit(real_stdout, line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
