#!/usr/bin/env python3
"""bench.py -- headline benchmark of the B200 BLS12-381 pairing path.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--dump-outputs DIR]

Workload (BASELINE.json configs[1]): a batch of 2^16 independent full pairings (Miller loop + final
exponentiation) per GPU per step, on synthetic subgroup points generated on the device by the
engine's own wNAF kernels.  One "step" = one pass of the hot path over one batch.  N > 1: one rank
per GPU (torchrun), every rank runs its own 2^16 batch (weak scaling, no data-path collective);
`value` = pairings of all ranks / max-over-ranks device time.

The JSON line carries, besides the base contract: `roofline` (integer-multiply bound: algorithmic
MAC32/s against the IMAD.WIDE peak measured in the same run), `cpu_baseline` (the C oracle timed on
the host cores, rank 0, bounded sample), `e2e` (same metric through the host-buffer C-ABI call,
copies inside the timed region), `secondary` (BASELINE configs[2..4] at their stated sizes: sharded multi-Miller pairs/s, G1 wNAF muls/s,
G2 wNAF + G2Prepared).

`--impl reference` times the reference's CPU algorithm (the C restatement in oracle/ -- the Rust
crate cannot be built in this image) on all host threads, on a bounded sample per step.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path[:0] = [ROOT]

BATCH_LOG2 = 16
MAC32_PER_PAIRING = 20621 * 300          # SURVEY.md 8(d): 20 621 Fq mul/sq x 300 MAC32
MAC32_PER_G1_WNAF = 2577 * 300           # wNAF w=4 mul + batch normalisation
MAC32_PER_MM_PAIR = 4684 * 300           # multi-Miller per pair incl. on-the-fly prepare
MAC32_PER_G2_WNAF_PREP = 7992 * 300      # G2 wNAF w=4 + normalisation + G2Prepared::from_affine
HBM_BYTES_PER_PAIRING = 104 + 200 + 576  # G1Affine + G2Affine in, Fq12 out
SEED = 0x5DBE62598D313D76
DUMP_ROWS = 1 << 15                      # 2^15 GT elements x 144 words x 8 B = 37.7 MB per dump


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch-log2", type=int, default=BATCH_LOG2)
    ap.add_argument("--no-secondary", action="store_true")
    ap.add_argument("--mm-log2", type=int, default=20)
    ap.add_argument("--wnaf-log2", type=int, default=24)
    ap.add_argument("--g2-log2", type=int, default=20)
    ap.add_argument("--prep-log2", type=int, default=20)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-mgpu", action="store_true")
    ap.add_argument("--no-wnaf-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the pairings the last step computed (rank 0) to DIR/*.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the CUDA path; the reference arm times a host-sized sample")
    return args


# ------------------------------------------------------------------------------------------------
# reference arm: the CPU algorithm on the host cores (rank 0 only)
# ------------------------------------------------------------------------------------------------
def oracle_inputs(n):
    """n affine pairs for the CPU arms: small multiples of the generators built with the oracle."""
    sys.path[:0] = [os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")]
    import datagen as dg
    return dg.g1_affine_points(n, 101), dg.g2_affine_points(n, 202)


def cpu_pairings_per_s(sample, threads):
    sys.path[:0] = [os.path.join(ROOT, "oracle")]
    import oracle_lib as o
    p, q = oracle_inputs(sample)
    o.pairing(p[:threads], q[:threads], threads)          # warm-up (page in, spawn)
    t0 = time.perf_counter()
    o.pairing(p, q, threads)
    dt = time.perf_counter() - t0
    return sample / dt, dt


def cpu_secondary_baselines(threads, budget_s=3.0):
    """The reference's CPU algorithm (C restatement, all host threads) on bounded samples of BASELINE configs[2..4]:
    multi-Miller pairs/s, G1 wNAF + normalisation muls/s, G2 wNAF + normalisation + G2Prepared muls/s."""
    sys.path[:0] = [os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")]
    import datagen as dg
    import oracle_lib as o
    out = {}

    def sized(fn, unit_probe):
        """run fn(n) on a probe, then once more on a sample sized for ~budget_s of wall clock"""
        t0 = time.perf_counter(); fn(unit_probe); dt = time.perf_counter() - t0
        n = max(unit_probe, int(unit_probe * budget_s / max(dt, 1e-3)))
        t0 = time.perf_counter(); fn(n); dt = time.perf_counter() - t0
        return n, dt

    p, q = oracle_inputs(256)
    def mm(n):
        reps = (n + 255) // 256
        o.multi_miller_product(__import__("numpy").tile(p, (reps, 1))[:n], __import__("numpy").tile(q, (reps, 1))[:n], threads)
    n, dt = sized(mm, threads * 16)
    out["multi_miller_loop"] = {"value": n / dt, "unit": "pairs/s", "cores": threads, "kind": "port",
                                "sample": "product of %d pairs in %.1f s (per-thread partial products, oracle/bls_oracle.c)" % (n, dt)}
    b1, k = dg.g1_points(256, 303), dg.rand_scalars(256, 304, edge_cases=False)
    import numpy as np
    def g1(n):
        reps = (n + 255) // 256
        r = o.g1_op("wnaf", np.tile(b1, (reps, 1))[:n], k=np.tile(k, (reps, 1))[:n], threads=threads)
        o.g1_batch_normalization(r)
    n, dt = sized(g1, threads * 64)
    out["g1_wnaf_mul"] = {"value": n / dt, "unit": "scalar-muls/s", "cores": threads, "kind": "port",
                          "sample": "%d G1 wNAF multiplications (threaded) + batch_normalization (one thread, as in the crate) in %.1f s" % (n, dt)}
    b2 = dg.g2_points(128, 305)
    def g2(n):
        reps = (n + 127) // 128
        r = o.g2_op("wnaf", np.tile(b2, (reps, 1))[:n], k=np.tile(k[:128], (reps, 1))[:n], threads=threads)
        r = o.g2_batch_normalization(r)
        o.g2_prepare(o.g2_into_affine(r), threads)
    n, dt = sized(g2, threads * 16)
    out["g2_wnaf_mul_prepare"] = {"value": n / dt, "unit": "scalar-muls/s", "cores": threads, "kind": "port",
                                  "sample": "%d G2 wNAF multiplications + batch_normalization + G2Prepared in %.1f s" % (n, dt)}
    return out


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    sys.path[:0] = [os.path.join(ROOT, "oracle")]
    import oracle_lib as o
    threads = o.default_threads()
    p, q = oracle_inputs(max(threads * 8, 64))
    # size one step to ~2 s of wall clock
    t0 = time.perf_counter(); o.pairing(p, q, threads); probe = time.perf_counter() - t0
    per_s = len(p) / probe
    sample = max(threads, int(per_s * 2.0))
    p, q = oracle_inputs(sample)
    for _ in range(args.warmup):
        o.pairing(p[:max(threads, sample // 8)], q[:max(threads, sample // 8)], threads)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        o.pairing(p, q, threads)
    dt = time.perf_counter() - t0
    value = sample * args.steps / dt
    line = {
        "impl": "reference", "metric": "BLS12-381 pairings/sec", "value": value, "unit": "pairings/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64",
        "data": "synthetic",
        "config": {"workload": "batch of independent full pairings (BASELINE configs[1]), bounded sample of %d pairings per step" % sample,
                   "batch": sample},
        "cpu_baseline": {"value": value, "unit": "pairings/s", "cores": threads, "kind": "port",
                         "sample": "%d pairings per step x %d steps, C restatement of the reference (oracle/bls_oracle.c), %d pthreads" % (sample, args.steps, threads)},
        "e2e": {"value": value, "unit": "pairings/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------------------------
# clocks sampler (nvidia-smi during the timed region)
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.samples, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            f = [x.strip() for x in s.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); pw.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx), "power_w_max": max(pw), "samples": len(sm),
                "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
def make_inputs(eng, n, seed, torch, np):
    """P_i = [a_i] g1, Q_i = [b_i] g2 on the device with the engine's own kernels (wNAF + batch
    normalisation), as affine rows.  Scalars: SplitMix64 stream, rejection-sampled below r."""
    import pairing_b200._native as nat

    def splitmix(seed, count):
        with np.errstate(over="ignore"):
            idx = np.arange(1, count + 1, dtype=np.uint64)
            z = np.uint64(seed & (2**64 - 1)) + idx * np.uint64(0x9E3779B97F4A7C15)
            z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
            z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
            return z ^ (z >> np.uint64(31))

    def scalars(seed):
        k = splitmix(seed, 4 * n).reshape(n, 4)
        k[:, 3] &= np.uint64((1 << 62) - 1)        # < 2^254 < r: uniform enough for a throughput workload
        k[:, 0] |= np.uint64(2)
        return torch.from_numpy(k.view(np.int64)).to(eng.device)

    one = [0x760900000002fffd, 0xebf4000bc40c0002, 0x5f48985753c758ba, 0x77ce585370525745, 0x5c071a97a256ec6d, 0x15f65ec3fa80e493]
    g1x = [0x5cb38790fd530c16, 0x7817fc679976fff5, 0x154f95c7143ba1c1, 0xf0ae6acdf3d0e747, 0xedce6ecc21dbf440, 0x120177419e0bfb75]
    g1y = [0xbaac93d50ce72271, 0x8c22631a7918fd8e, 0xdd595f13570725ce, 0x51ac582950405194, 0x0e1c8c3fad0059c0, 0x0bbc3efc5008a26a]
    g2 = [[0xf5f28fa202940a10, 0xb3f5fb2687b4961a, 0xa1a893b53e2ae580, 0x9894999d1a3caee9, 0x6f67b7631863366b, 0x058191924350bcd7],
          [0xa5a9c0759e23f606, 0xaaa0c59dbccd60c3, 0x3bb17e18e2867806, 0x1b1ab6cc8541b367, 0xc2b6ed0ef2158547, 0x11922a097360edf3],
          [0x4c730af860494c4a, 0x597cfa1f5e369c5a, 0xe7e6856caa0a635a, 0xbbefb5e96e0d495f, 0x07d3a975f0ef25a2, 0x0083fd8e7e80dae5],
          [0xadc0fc92df64b05d, 0x18aa270a2b1461dc, 0x86adac6a3be4eba0, 0x79495c4ec93da33a, 0xe7175850a43ccaed, 0x0b2bc2a163de1bf2]]
    b1 = np.array([g1x + g1y + one], dtype=np.uint64)
    b2 = np.array([g2[0] + g2[1] + g2[2] + g2[3] + one + [0] * 6], dtype=np.uint64)
    base1 = torch.from_numpy(np.repeat(b1, n, 0).view(np.int64)).to(eng.device)
    base2 = torch.from_numpy(np.repeat(b2, n, 0).view(np.int64)).to(eng.device)
    p = eng.g1_wnaf_mul(base1, scalars(seed ^ 0x1111))
    q = eng.g2_wnaf_mul(base2, scalars(seed ^ 0x2222))
    eng.g1_batch_normalization_(p)
    eng.g2_batch_normalization_(q)
    pa = eng.jacobian_to_affine_rows(p, 6)
    qa = eng.jacobian_to_affine_rows(q, 12)
    torch.cuda.synchronize()
    assert pa.shape[1] == nat.W_G1A and qa.shape[1] == nat.W_G2A
    return pa, qa, p, scalars(seed ^ 0x3333)


def dump_outputs(dirname, out, np):
    """Write the (n, 72) GT elements of one step as DIR/pairing.npy: the rows of a fixed, seeded sample of at most
    DUMP_ROWS pairings (every row of a smaller batch), each as its 144 32-bit words (12 Fq coefficients x 12 Montgomery
    limbs, least significant first), in float64, which holds every word exactly.  DIR/pairing_rows.npy: the row indices."""
    n = out.shape[0]
    rows = np.sort(np.random.default_rng(SEED).choice(n, min(n, DUMP_ROWS), replace=False))
    words = out.cpu().numpy()[rows].view(np.uint32)
    os.makedirs(dirname, exist_ok=True)
    np.save(os.path.join(dirname, "pairing.npy"), words.astype(np.float64))
    np.save(os.path.join(dirname, "pairing_rows.npy"), rows.astype(np.float64))


def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world != args.gpus and world != 1:
        raise SystemExit("WORLD_SIZE=%d does not match --gpus %d" % (world, args.gpus))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    from pairing_b200.device import DeviceEngine
    eng = DeviceEngine(device=local_rank)
    ctx = eng.ctx
    n = 1 << args.batch_log2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=eng.device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    pa, qa, g1_jac, g1_scalars = make_inputs(eng, n, SEED + rank, torch, np)
    out = torch.empty((n, 72), dtype=torch.int64, device=eng.device)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=eng.device)   # > 126 MB L2

    def step():
        flush.zero_()                       # evict the previous step's inputs/outputs from L2
        eng.pairing(pa, qa, out)

    # integer-multiply peak in the same run (roofline denominator)
    peak_macs, _ = ctx.imad_peak(0, 4000)
    fpmul_macs, _ = ctx.imad_peak(1, 2000)

    for _ in range(max(args.warmup, 1)):
        step()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = ctx.launch_count
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    ev0.record()
    for i in range(args.steps):
        flush.zero_()
        kev[i][0].record()
        eng.pairing(pa, qa, out)
        kev[i][1].record()
    ev1.record()
    barrier()
    launches = ctx.launch_count - launches0
    total_ms = max_over_ranks(ev0.elapsed_time(ev1))
    kernel_ms = sum(a.elapsed_time(b) for a, b in kev) / args.steps     # the pairing kernel alone, this rank
    clocks = sampler.stop() if rank == 0 else None
    value = world * n * args.steps / (total_ms * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, out, np)               # `out` holds the last timed step's result

    # ---- e2e: host buffers through the C-ABI call a user makes (copies inside the timed region)
    ph = torch.empty(pa.shape, dtype=torch.int64).pin_memory(); ph.copy_(pa.cpu())
    qh = torch.empty(qa.shape, dtype=torch.int64).pin_memory(); qh.copy_(qa.cpu())
    oh = torch.empty((n, 72), dtype=torch.int64).pin_memory()
    import ctypes
    lib = ctx._lib

    def e2e_step():
        rc = lib.bls_pairing_batch(ctx._ctx, ph.data_ptr(), qh.data_ptr(), oh.data_ptr(), n)
        if rc != 0:
            raise SystemExit("bls_pairing_batch failed: %d" % rc)
    e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        e2e_step()
    e2e_dt = max_over_ranks(time.perf_counter() - t0)
    e2e_value = world * n * args.steps / e2e_dt
    checksum = int(oh[:, 0].sum().item()) & 0xFFFFFFFF            # the step's result is read on the host
    same = bool(torch.equal(oh, out.cpu()))                       # e2e output == device-path output

    # ---- secondary: the other BASELINE configs at their stated sizes (one warm-up on a slice, one timed pass each;
    # inputs are the 2^16 distinct points/scalars tiled to size -- the arithmetic does not depend on the values)
    secondary = {}
    if not args.no_secondary:
        def tile(t, m):
            return t.repeat((m + t.shape[0] - 1) // t.shape[0], 1)[:m].contiguous()

        def timed(fn):
            barrier()
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record(); r = fn(); t1.record()
            barrier()
            return max_over_ranks(t0.elapsed_time(t1)), r

        def entry(units, ms, mac_per_unit, **kw):
            rate = world * units / (ms * 1e-3)
            d = {"value": rate, "units_per_gpu": units, "ms": ms, "roofline_frac": rate / world * mac_per_unit / peak_macs}
            d.update(kw)
            return d

        # configs[0]: a single pairing e(P, Q) (latency of a batch of one) and the crate's bench_pairing_full shape (1000 pairings)
        one_out = torch.empty((1, 72), dtype=torch.int64, device=eng.device)
        eng.pairing(pa[:1].contiguous(), qa[:1].contiguous(), one_out)
        ms_one, _ = timed(lambda: eng.pairing(pa[:1].contiguous(), qa[:1].contiguous(), one_out))
        k_out = torch.empty((1000, 72), dtype=torch.int64, device=eng.device)
        eng.pairing(pa[:1000].contiguous(), qa[:1000].contiguous(), k_out)
        ms_k, _ = timed(lambda: eng.pairing(pa[:1000].contiguous(), qa[:1000].contiguous(), k_out))
        # the crate's bench_pairing_full calls pairing on PROJECTIVE points: into_affine of both arguments inside the call
        pj1 = g1_jac[:1000].contiguous()
        qj1 = torch.zeros((1000, 36), dtype=torch.int64, device=eng.device)
        qj1[:, :24] = qa[:1000, :24]; qj1[:, 24:30] = g1_jac[:1, 12:18]
        eng.pairing_projective(pj1[:1].contiguous(), qj1[:1].contiguous(), one_out)
        ms_one_proj, _ = timed(lambda: eng.pairing_projective(pj1[:1].contiguous(), qj1[:1].contiguous(), one_out))
        ms_k_proj, _ = timed(lambda: eng.pairing_projective(pj1, qj1, k_out))
        secondary["single_pairing"] = {"latency_ms": ms_one, "batch_1000_ms": ms_k, "projective_inputs_latency_ms": ms_one_proj, "projective_inputs_batch_1000_ms": ms_k_proj, "value": world * 1000 / (ms_k * 1e-3), "unit": "pairings/s",
                                       "units_per_gpu": 1000, "ms": ms_k, "roofline_frac": 1000 / (ms_k * 1e-3) * MAC32_PER_PAIRING / peak_macs,
                                       "config": "configs[0]: one pairing and the 1000 pairings of bench_pairing_full, on the warp-cooperative kernel (one WARP per pairing)"}
        # the signature-verification shape: final_exponentiation(miller_loop(a FEW pairs)) in one call -- Miller loops one warp per
        # pair, fold and final exponentiation in the tail kernel (latency path), against the lane-pair multi-Miller kernel
        prod_ms = {}
        for npairs in (2, 64):
            pp, qq = pa[:npairs].contiguous(), qa[:npairs].contiguous()
            eng.pairing_product(pp, qq)
            prod_ms["n%d_ms" % npairs], _ = timed(lambda: eng.pairing_product(pp, qq))
        ctx.set_latency_path_limits(0, 0)
        eng.pairing_product(pa[:2].contiguous(), qa[:2].contiguous())
        prod_ms["n2_lane_pair_kernels_ms"], _ = timed(lambda: eng.pairing_product(pa[:2].contiguous(), qa[:2].contiguous()))
        ctx.set_latency_path_limits(2560, 2560)
        secondary["pairing_product_small"] = dict(prod_ms, value=world * 2 / (prod_ms["n2_ms"] * 1e-3), unit="pairings/s", units_per_gpu=2, ms=prod_ms["n2_ms"],
                                                  config="one bls_pairing_product_dev call over 2 / 64 pairs (batch-verification of a single signature: a product of two pairings)")
        from pairing_b200 import dist as pdist
        # configs[2] as stated: ONE multi_miller_loop product of 2^20 pairs IN TOTAL, sharded over the ranks (strong scaling),
        # with one shared final exponentiation.  Per rank: Miller kernel (one partial per block) + fold to one 576-byte
        # partial; all-gather (NCCL); fold of the `world` partials + the final exponentiation on the warp-cooperative engine.
        nm = 1 << args.mm_log2
        lo, hi = pdist.shard_range(nm, rank, world)
        pm, qm = tile(pa, hi - lo), tile(qa, hi - lo)
        pdist.pairing_product_sharded(eng, pm[:4096].contiguous(), qm[:4096].contiguous())
        eng._buf("mm", ctx.multi_miller_scratch_bytes(hi - lo))     # grow-only scratch sized before the timed passes
        def mm_run():
            return pdist.pairing_product_sharded(eng, pm, qm)[0]
        mm_run()                                                    # one untimed full-size pass, then the mean of three
        ms3, fe = timed(lambda: [mm_run() for _ in range(3)][-1])
        ms = ms3 / 3
        # the same product once more with an event after every phase (this rank's times; max over ranks below)
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        barrier()
        ev[0].record()
        part = eng.multi_miller_loop(pm, qm)
        ev[1].record()
        allp = pdist.all_gather_partials(part) if world > 1 else part
        ev[2].record()
        fe2, ok2 = eng.fq12_product_tail(allp, final_exp=True)
        ev[3].record()
        barrier()
        phases = [max_over_ranks(ev[i].elapsed_time(ev[i + 1])) for i in range(3)]
        assert bool(torch.equal(fe, fe2)) and int(ok2.item()) == 1
        rate = nm / (ms * 1e-3)
        secondary["multi_miller_loop"] = {
            "value": rate, "unit": "pairs/s", "pairs_total": nm, "pairs_per_gpu": hi - lo, "ms": ms, "passes": 3, "scaling": "strong",
            "roofline_frac": rate / world * MAC32_PER_MM_PAIR / peak_macs,
            "phase_ms": {"miller_and_fold_per_gpu": phases[0], "all_gather": phases[1], "fold_and_final_exponentiation": phases[2]},
            "collective": "all_gather of one 576-byte Fq12 per rank (NCCL)" if world > 1 else "none (1 rank)",
            "gt_checksum": int(fe.cpu().numpy().view(np.uint64).sum(dtype=np.uint64)) & 0xFFFFFFFF,
            "config": "configs[2]: ONE product of 2^%d pairs sharded over %d GPU(s) + one final exponentiation" % (args.mm_log2, world)}
        del pm, qm
        # configs[3]: G1 wNAF scalar multiplication of 2^24 points per GPU + batch affine normalisation
        nw = 1 << args.wnaf_log2
        bases, ks = tile(g1_jac, nw), tile(g1_scalars, nw)
        wout = torch.empty_like(bases)
        eng.g1_batch_normalization_(eng.g1_wnaf_mul(bases[:4096].contiguous(), ks[:4096].contiguous(), 0))
        eng._buf("bn", ctx.batch_normalization_scratch_bytes(1, nw))
        ms_mul, _ = timed(lambda: eng.g1_wnaf_mul(bases, ks, 0, wout))
        ms_norm, _ = timed(lambda: eng.g1_batch_normalization_(wout))
        secondary["g1_wnaf_mul"] = entry(nw, ms_mul + ms_norm, MAC32_PER_G1_WNAF, unit="scalar-muls/s", ms_wnaf=ms_mul, ms_normalise=ms_norm,
                                         config="configs[3]: 2^%d points x 255-bit scalars per GPU, wNAF w=4 + batch_normalization" % args.wnaf_log2)
        # the same through the host-buffer C-ABI calls (pinned buffers): chunked H2D / kernel / D2H pipeline + normalisation
        if not args.no_wnaf_e2e:
            bh = torch.empty(bases.shape, dtype=torch.int64).pin_memory(); bh.copy_(bases)
            kh = torch.empty(ks.shape, dtype=torch.int64).pin_memory(); kh.copy_(ks)
            oh2 = torch.empty(bases.shape, dtype=torch.int64).pin_memory()
            torch.cuda.synchronize()
            def wnaf_e2e():
                rc = ctx._lib.bls_g1_wnaf_mul_batch(ctx._ctx, bh.data_ptr(), kh.data_ptr(), oh2.data_ptr(), nw)
                rc = rc or ctx._lib.bls_g1_batch_normalization(ctx._ctx, oh2.data_ptr(), nw)
                if rc != 0:
                    raise SystemExit("g1 wnaf e2e failed: %d" % rc)
            wnaf_e2e()
            barrier()
            t0 = time.perf_counter(); wnaf_e2e(); dt = max_over_ranks(time.perf_counter() - t0)
            secondary["g1_wnaf_mul"]["e2e"] = {"value": world * nw / dt, "unit": "scalar-muls/s", "ms": dt * 1e3,
                                               "h2d_bytes": nw * (144 + 32) + nw * 144, "d2h_bytes": 2 * nw * 144,
                                               "api": "bls_g1_wnaf_mul_batch + bls_g1_batch_normalization (host buffers, pinned)",
                                               "matches_device_path": bool(torch.equal(oh2[:: 4099], wout[:: 4099].cpu()))}
            del bh, kh, oh2
        del bases, ks, wout
        # configs[4]: G2 wNAF scalar multiplication + batch normalisation + G2Prepared precomputation, 2^20 points per GPU
        n2 = 1 << args.g2_log2
        one = g1_jac[:1, 12:18]
        q2 = torch.zeros((n, 36), dtype=torch.int64, device=eng.device)
        q2[:, :24] = qa[:, :24]; q2[:, 24:30] = one
        b2, k2 = tile(q2, n2), tile(g1_scalars, n2)
        w2 = torch.empty_like(b2)
        eng.g2_batch_normalization_(eng.g2_wnaf_mul(b2[:4096].contiguous(), k2[:4096].contiguous(), 0))
        eng._buf("bn", ctx.batch_normalization_scratch_bytes(2, n2))
        ms_mul, _ = timed(lambda: eng.g2_wnaf_mul(b2, k2, 0, w2))
        ms_norm, _ = timed(lambda: eng.g2_batch_normalization_(w2))
        aff2 = eng.jacobian_to_affine_rows(w2, 12)
        del b2, k2, w2
        npre = min(n2, 1 << args.prep_log2)                         # default: all 2^20 points (20.5 GB of coefficients)
        prep = torch.empty((npre, 68 * 36 + 1), dtype=torch.int64, device=eng.device)
        eng.g2_prepare(aff2[:4096].contiguous(), prep[:4096])
        ms_prep, _ = timed(lambda: eng.g2_prepare(aff2[:npre], prep))
        ms_prep_full = ms_prep * n2 / npre
        secondary["g2_wnaf_mul_prepare"] = entry(n2, ms_mul + ms_norm + ms_prep_full, MAC32_PER_G2_WNAF_PREP, unit="scalar-muls/s",
                                                 ms_wnaf=ms_mul, ms_normalise=ms_norm, ms_prepare=ms_prep_full, prepared_points_timed=npre,
                                                 config="configs[4]: 2^%d G2 points per GPU: wNAF w=4 + batch_normalization + G2Prepared (19 592 B per point)" % args.g2_log2)
        del prep, aff2

        # rows of SURVEY 8(f) built this round, at moderate sizes (one warm-up, one timed pass)
        nf = 1 << 20
        wfix = 16                                                   # recommended_wnaf_for_num_scalars(2^20), ec.rs:907-921
        fb = g1_jac[5:6].contiguous()
        ms_tab, table = timed(lambda: eng.wnaf_table(fb, wfix))
        kf = tile(g1_scalars, nf)
        fout = torch.empty((nf, 18), dtype=torch.int64, device=eng.device)
        eng.wnaf_fixed_base(table, wfix, kf[:4096].contiguous())
        ms_fix, _ = timed(lambda: eng.wnaf_fixed_base(table, wfix, kf, out=fout))
        secondary["g1_wnaf_fixed_base"] = entry(nf, ms_fix, (254 * 7 + 14 * 16) * 300, unit="scalar-muls/s", window=wfix, ms_table=ms_tab,
                                               config="SURVEY 8f-1: Wnaf::base(g, 2^20).scalar(s): one 2^15-entry table, 2^20 scalars per GPU")
        del kf, fout, table
        # 2^16 pairings against ONE prepared G2 point (coefficients staged in shared memory by a TMA bulk copy)
        q1p = eng.g2_prepare(qa[:1].contiguous())
        sq_out = torch.empty((n, 72), dtype=torch.int64, device=eng.device)
        eng.pairing_shared_q(pa, q1p, sq_out)
        ms_sq, _ = timed(lambda: eng.pairing_shared_q(pa, q1p, sq_out))
        secondary["pairing_shared_q"] = entry(n, ms_sq, (5156 + 13705) * 300, unit="pairings/s",
                                             config="2^%d pairings e(P_i, Q) per GPU against one G2Prepared (fixed-key verification shape)" % args.batch_log2)
        npow = 1 << 14
        gt = out[:npow].contiguous()
        eng.fq12_pow(gt[:256].contiguous(), g1_scalars[:256].contiguous())
        ms_pow, _ = timed(lambda: eng.fq12_pow(gt, g1_scalars[:npow].contiguous()))
        secondary["gt_pow"] = entry(npow, ms_pow, (254 * 36 + 127 * 54) * 300, unit="powers/s",
                                    config="SURVEY 8f-4: Fq12::pow(FrRepr) for 2^14 GT elements per GPU")
        # SURVEY 8f-2: G1Compressed::into_affine (checked: square root, lexicographic y, subgroup test) through the host-buffer
        # call -- bytes in host memory, affine rows + status back; wall clock around the call, H2D and D2H included
        ndec = 1 << 18
        dec_aff = np.ascontiguousarray(tile(pa, ndec).cpu().numpy().view(np.uint64))
        dec_bytes = eng.ctx.encode(False, dec_aff, True)
        import pairing_b200._native as nat
        dec_buf = np.frombuffer(dec_bytes, dtype=np.uint8).copy()
        dec_back, dec_status = np.zeros((ndec, 13), dtype=np.uint64), np.zeros(ndec, dtype=np.uint8)
        def decode_call(count):
            eng.ctx._check(eng.ctx._lib.bls_g1_decode_batch(eng.ctx._ctx, nat._p(dec_buf), 1, 1, nat._p(dec_back), nat._p(dec_status), count))
        decode_call(4096)
        barrier()
        t0 = time.perf_counter()
        decode_call(ndec)
        ms_dec = max_over_ranks((time.perf_counter() - t0) * 1e3)
        barrier()
        secondary["g1_decode_compressed_checked"] = entry(ndec, ms_dec, 4514 * 300, unit="points/s", round_trip=bool(np.array_equal(dec_back, dec_aff)) and not dec_status.any(),
                                                          config="SURVEY 8f-2: 2^18 compressed G1 points per GPU decoded with curve and subgroup validation (ec.rs:760-868), host buffers; 4514 M per point is the reference's count (sqrt + multiplication by r), the kernel decides the subgroup with the endomorphism test")
        del dec_aff, dec_bytes, dec_back, dec_buf
        # the same for 2^16 compressed G2 points (Fq2 square root by Algorithm 9 of eprint 2012/685, psi(Q) = [u]Q as the subgroup test)
        ndec2 = 1 << 16
        dec_aff2 = np.ascontiguousarray(tile(qa, ndec2).cpu().numpy().view(np.uint64))
        dec_buf2 = np.frombuffer(eng.ctx.encode(True, dec_aff2, True), dtype=np.uint8).copy()
        dec_back2, dec_status2 = np.zeros((ndec2, 25), dtype=np.uint64), np.zeros(ndec2, dtype=np.uint8)
        def decode2_call(count):
            eng.ctx._check(eng.ctx._lib.bls_g2_decode_batch(eng.ctx._ctx, nat._p(dec_buf2), 1, 1, nat._p(dec_back2), nat._p(dec_status2), count))
        decode2_call(2048)
        barrier()
        t0 = time.perf_counter()
        decode2_call(ndec2)
        ms_dec2 = max_over_ranks((time.perf_counter() - t0) * 1e3)
        barrier()
        secondary["g2_decode_compressed_checked"] = {"value": world * ndec2 / (ms_dec2 * 1e-3), "unit": "points/s", "units_per_gpu": ndec2, "ms": ms_dec2,
                                                     "round_trip": bool(np.array_equal(dec_back2, dec_aff2)) and not dec_status2.any(),
                                                     "config": "SURVEY 8f-2: 2^16 compressed G2 points per GPU decoded with curve and subgroup validation (ec.rs:1419-1540), host buffers"}
        del dec_aff2, dec_buf2, dec_back2
        # SURVEY 8f-3: CurveProjective::mul_assign (double-and-add, ec.rs:534-553) for 2^18 G1 points through the host-buffer call
        nmul = 1 << 18
        mul_b = np.ascontiguousarray(tile(g1_jac, nmul).cpu().numpy().view(np.uint64))
        mul_k = np.ascontiguousarray(tile(g1_scalars, nmul).cpu().numpy().view(np.uint64))
        eng.ctx.g1_mul(mul_b[:4096], mul_k[:4096])
        barrier()
        t0 = time.perf_counter()
        eng.ctx.g1_mul(mul_b, mul_k)
        ms_mul = max_over_ranks((time.perf_counter() - t0) * 1e3)
        barrier()
        secondary["g1_mul_assign"] = entry(nmul, ms_mul, (254 * 7 + 127 * 16) * 300, unit="scalar-muls/s",
                                           config="SURVEY 8f-3: mul_assign (double-and-add over the 255-bit scalar) for 2^18 G1 points per GPU, host buffers (wall clock, copies and the Python wrapper's allocations included)")
        del mul_b, mul_k

    # host copies for the single-process multi-device measurement below (rank 0 only)
    mg_host = None
    if rank == 0 and not args.no_secondary and not args.no_mgpu:
        nm = 1 << args.mm_log2
        reps = (nm + n - 1) // n
        mg_host = (torch.empty((nm, pa.shape[1]), dtype=torch.int64).pin_memory(), torch.empty((nm, qa.shape[1]), dtype=torch.int64).pin_memory())
        mg_host[0].copy_(pa.cpu().repeat(reps, 1)[:nm]); mg_host[1].copy_(qa.cpu().repeat(reps, 1)[:nm])

    if world > 1:
        dist.barrier()
        torch.cuda.synchronize()
        dist.destroy_process_group()
    if rank != 0:
        return 0

    # ---- configs[2] through the C ABI a Rust / C caller binds: ONE process, ONE call, all `world` devices
    # (bls_mgpu_pairing_product: host buffers in, one GT element out; H2D, per-device Miller kernels, peer-copy gather,
    # fold + final exponentiation inside the call).  The other ranks have left; their devices are idle.
    if mg_host is not None:
        import pairing_b200._native as nat
        if world > 1:
            time.sleep(2.0)                                         # let the other ranks' processes tear down
        try:
            with nat.MultiGpu(world) as mg:
                nm = mg_host[0].shape[0]
                lib = mg._lib
                gt = np.zeros((1, 72), dtype=np.uint64); ok = np.zeros(1, dtype=np.uint8)
                def mg_run():
                    rc = lib.bls_mgpu_pairing_product(mg._m, mg_host[0].data_ptr(), mg_host[1].data_ptr(), nm, gt.ctypes.data, ok.ctypes.data)
                    if rc != 0:
                        raise RuntimeError("bls_mgpu_pairing_product failed: %d" % rc)
                mg_run()
                best, phases = None, None
                for _ in range(3):
                    t0 = time.perf_counter(); mg_run(); dt = time.perf_counter() - t0
                    if best is None or dt < best:
                        best, phases = dt, mg.last_phase_ms()
                secondary["multi_miller_loop"]["e2e_c_abi"] = {
                    "value": nm / best, "unit": "pairs/s", "ms": best * 1e3, "devices": world, "api": "bls_mgpu_pairing_product (one process, host buffers, pinned)",
                    "h2d_bytes": nm * (104 + 200), "d2h_bytes": 577, "phase_ms": phases, "is_some": int(ok[0]),
                    "gt_checksum": int(gt.sum(dtype=np.uint64)) & 0xFFFFFFFF}
        except Exception as e:                                      # reported, never fatal for the headline line
            secondary["multi_miller_loop"]["e2e_c_abi"] = {"error": str(e)[:200]}

    # ---- CPU baseline on the host cores (bounded sample)
    cpu = None
    if not args.no_cpu_baseline:
        threads = len(os.sched_getaffinity(0))
        probe_rate, _ = cpu_pairings_per_s(max(threads * 4, 32), threads)
        sample = max(threads, int(probe_rate * 10.0))             # ~10 s of host work
        rate, dt = cpu_pairings_per_s(sample, threads)
        cpu = {"value": rate, "unit": "pairings/s", "cores": threads, "kind": "port",
               "sample": "%d full pairings of the same workload in %.1f s, C restatement of the reference (oracle/bls_oracle.c), %d pthreads" % (sample, dt, threads)}
        if secondary:
            for key, base in cpu_secondary_baselines(threads).items():
                if key in secondary:
                    secondary[key]["cpu_baseline"] = base

    traffic, executed = None, None                                  # per launch of the dominant kernel, from the committed ncu capture
    try:
        prof = json.load(open(os.path.join(ROOT, "profiles", "r2_pair_miller.json")))
        if n == prof["n_pairings"]:
            traffic = prof["traffic_bytes_per_launch"]
        executed = prof["executed_wide_mac32_per_pairing"]
    except Exception:
        pass
    kernel_rate = n / (kernel_ms * 1e-3)                          # pairings/s of the dominant kernel on this GPU
    achieved = kernel_rate * MAC32_PER_PAIRING
    line = {
        "metric": "BLS12-381 pairings/sec", "value": value, "unit": "pairings/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 1), "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u32", "data": "synthetic",
        "config": {"workload": "batch of 2^%d independent full pairings per GPU (Miller loop + final exponentiation), BASELINE configs[1]" % args.batch_log2,
                   "batch_per_gpu": n, "inputs": "G1Affine/G2Affine subgroup points = seeded scalar multiples of the generators, resident in HBM",
                   "l2": "256 MiB buffer written between timed iterations (L2 flush)",
                   "arithmetic": "Fq as 12 x 32-bit Montgomery limbs, IMAD.WIDE.U32 carry chains, bit-exact with the reference", "parallelism": "dp%d, no data-path collective" % world},
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "pairings/s", "h2d_bytes_per_step": n * (104 + 200), "d2h_bytes_per_step": n * 576,
                "api": "bls_pairing_batch (host buffers, pinned)", "matches_device_path": same, "checksum": checksum},
        "gpu_launches": int(launches),
        "roofline": {"bound": "imad", "achieved": achieved / 1e12, "peak": peak_macs / 1e12, "unit": "TMAC32/s",
                     "frac": achieved / peak_macs, "traffic": traffic,
                     "frac_note": "ALGORITHMIC MAC32 (the reference algorithm's 20 621 Fq products x 300, SURVEY 8d) over the measured peak; the kernel EXECUTES fewer multiplies (cyclotomic squarings, dedicated Fq squaring): see executed_mac32_per_pairing / frac_executed",
                     "executed_mac32_per_pairing": executed,
                     "frac_executed": (kernel_rate * executed / peak_macs) if executed else None,
                     "traffic_note": "bytes per launch, dram__bytes_read.sum + dram__bytes_write.sum of profiles/r2_pair_miller.md; mostly local-memory write-back, ~53 GB/s; algorithmic bytes are 57.7 MB per launch",
                     "kernel": "k_pair_miller<true> (fused Miller loop + final exponentiation on lane pairs, one launch per step)",
                     "kernel_ms": kernel_ms, "mac32_per_pairing": MAC32_PER_PAIRING,
                     "peak_source": "chain of dependent IMAD.WIDE.U32 (bls_imad_peak variant 0, SASS-checked by tests/test_abi.py) measured in this run: one 32x32->64 multiply per 4 cycles per SM sub-partition; MEASURED_PEAKS.json has no integer figure",
                     "fp_mul_chain_tmac32": fpmul_macs / 1e12,
                     "hbm": {"achieved_gbs": kernel_rate * HBM_BYTES_PER_PAIRING / 1e9, "note": "algorithmic bytes; far from the 6548.8 GB/s measured HBM peak: the path is integer-multiply bound"}},
        "cpu_baseline": cpu,
        "secondary": secondary,
    }
    print(json.dumps(line))
    return 0


def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
