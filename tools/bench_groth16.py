"""Groth16 proving (bls_groth16_prove_dev through DeviceEngine.groth16_prove) on one GPU.
Shapes: m = 1 proof at len = 2^16, 2^20 and 2^22; m = 4 at 2^20; m = 64 at 2^12; each with num_aux = len - 4 and 4 inputs,
densities drawn with a fixed seed (a_aux 90 %, b_input all set, b_aux 50 %).  The queries are bench.make_inputs' 2^20
subgroup points, repeated where a query is longer.
Each shape is timed by CUDA events as the median of --reps launches after one warm-up, with a 256 MiB write between
launches (as bench.py does).  In the same process the script times the standalone calls the prove call contains, run back
to back: groth16_h and the five msm_batch calls at the same lengths.  A separate torch.profiler pass per shape (one call,
after the timed ones) gives the GPU time of k_groth16_gather and of the tail kernels k_groth16_mul + k_groth16_assemble.
    python tools/bench_groth16.py --out groth16_prove.json
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT]

SHAPES = ((16, 1), (20, 1), (22, 1), (20, 4), (12, 64))
NUM_INPUTS = 4


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=7)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_groth16.py needs a CUDA device")
    import bench
    import pairing_b200._native as nat
    from pairing_b200.device import DeviceEngine
    eng = DeviceEngine(device=0)
    gpu = {"name": torch.cuda.get_device_name(0)}
    try:
        gpu["nvidia_smi"] = subprocess.check_output(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv"],
                                                    text=True).strip().splitlines()[-1]
    except Exception as e:                                    # noqa: BLE001 -- recorded, not fatal
        gpu["nvidia_smi"] = "unavailable: %s" % e
    pa, qa, _, _ = bench.make_inputs(eng, 1 << 20, 0x3A5E, torch, np)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=eng.device)
    gen = torch.Generator(device=eng.device).manual_seed(0x6016)
    rng = np.random.default_rng(0x6016)

    def timed(fn):
        fn()
        ts = []
        for _ in range(args.reps):
            flush.fill_(1)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            b.synchronize()
            ts.append(a.elapsed_time(b))
        return sorted(ts)[len(ts) // 2]

    def query(pts, count):
        return pts[torch.arange(count, device=eng.device) % pts.shape[0]].contiguous()

    def scalars(*shape):
        x = torch.randint(-(1 << 63), (1 << 63) - 1, shape + (4,), dtype=torch.int64, device=eng.device, generator=gen)
        x[..., 3] &= (1 << 60) - 1                            # canonical: < 2^252 < r
        return x

    vk1, vk2 = pa[:3].cpu().numpy().view(np.uint64), qa[:2].cpu().numpy().view(np.uint64)
    rows = []
    for lg, m in SHAPES:
        length = 1 << lg
        ni, na = NUM_INPUTS, length - NUM_INPUTS
        dens = (rng.random(na) < 0.9, np.ones(ni, dtype=bool), rng.random(na) < 0.5)
        la, lb = ni + int(dens[0].sum()), int(dens[1].sum() + dens[2].sum())
        params = nat.Groth16Params(vk1[0], vk1[1], vk1[2], vk2[0], vk2[1], query(pa, length - 1), query(pa, na), query(pa, la), query(pa, lb),
                                   query(qa, lb))
        a, b, c = scalars(m, length), scalars(m, length), scalars(m, length)
        inp, aux, r, s = scalars(m, ni), scalars(m, na), scalars(m), scalars(m)
        out = torch.empty((m, nat.W_PROOF), dtype=torch.int64, device=eng.device)
        h_out = torch.empty((m, length - 1, 4), dtype=torch.int64, device=eng.device)
        ks = {"l": scalars(m, na), "a": scalars(m, la), "b": scalars(m, lb)}
        sums = {g2: torch.empty((m, nat.W_G2 if g2 else nat.W_G1), dtype=torch.int64, device=eng.device) for g2 in (False, True)}

        def prove():
            eng.groth16_prove(params, a, b, c, inp, aux, dens, r, s, out=out)

        def parts():
            eng.groth16_h(a, b, c, out=h_out)
            eng.msm_batch(params.h, h_out, out=sums[False])
            eng.msm_batch(params.l, ks["l"], out=sums[False])
            eng.msm_batch(params.a, ks["a"], out=sums[False])
            eng.msm_batch(params.b_g1, ks["b"], out=sums[False])
            eng.msm_batch(params.b_g2, ks["b"], g2=True, out=sums[True])

        ms_prove = timed(prove)
        ms_parts = timed(parts)
        flush.fill_(1)
        torch.cuda.synchronize()
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            prove()
            torch.cuda.synchronize()
        kern = {}
        for ev in prof.key_averages():
            for k in ("k_groth16_gather", "k_groth16_mul", "k_groth16_assemble"):
                if k in ev.key:
                    kern[k] = kern.get(k, 0.0) + ev.self_device_time_total / 1e3
        rows.append({"log_len": lg, "m": m, "num_inputs": ni, "num_aux": na, "a_len": la, "b_len": lb, "ms_prove": ms_prove,
                     "ms_parts": ms_parts, "ratio": ms_prove / ms_parts, "ms_per_proof": ms_prove / m,
                     "ms_gather": kern.get("k_groth16_gather"), "ms_mul": kern.get("k_groth16_mul"),
                     "ms_assemble": kern.get("k_groth16_assemble")})
        print(json.dumps(rows[-1]), flush=True)
        del params, a, b, c, inp, aux, r, s, out, h_out, ks, sums
        eng._scratch.clear()
        torch.cuda.empty_cache()
    res = {"gpu": gpu, "reps": args.reps, "flush_bytes": 256 << 20,
           "inputs": "torch.randint limbs, top limb masked to 60 bits (canonical); queries: bench.make_inputs(eng, 2^20, 0x3A5E) repeated",
           "rows": rows}
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
