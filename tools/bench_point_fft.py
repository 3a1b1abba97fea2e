"""The point FFT and FK20 on one GPU: bls_g1_fft_dev, bls_g2_fft_dev and bls_kzg_open_all_dev (through DeviceEngine).
Shapes: G1 fft and ifft at 1 x 2^16, 1 x 2^20 and 64 x 2^12, G2 fft at 1 x 2^16; kzg_open_all at n = 2^12 with m = 1 and
m = 64, and at n = 2^16 with m = 1.
Each transform is timed alternately, in the same process, with bls_g*_wnaf_mul_dev over as many (point, scalar) pairs as the
transform has non-trivial multiplications: per row, sum over the stages s of (n / 2^(s+1)) (2^s - 1) = L n / 2 - (n - 1)
butterflies with a twiddle other than one, plus n for the scaling of ifft (and of the coset kinds).  Both are reported per
multiplication.  The wNAF pairs are bench.make_inputs' points as Jacobian rows and torch.randint scalars with the top limb
masked to 62 bits (254-bit, canonical: the twiddles are 255-bit integers).
kzg_open_all at n = 2^12 and m = 4 is timed alternately with the chain it replaces: bls_kzg_open_dev over the 4 polynomials
each replicated n times with z = omega^k (2^14 openings, 2^26 coefficients: the open call's limit); the outputs are compared.
Points are bench.make_inputs' 2^20 subgroup points (repeated); coefficients are torch.randint limbs with the top limb masked
to 60 bits.  Each call is timed by CUDA events as the median of --reps launches after one warm-up, with a 256 MiB write
between launches (the L2 holds nothing of the previous launch).  The card's name and nvidia-smi's power limit are recorded in
the same run.
    python tools/bench_point_fft.py --out point_fft.json
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")]

FFT_SHAPES = ((False, "fft", 1, 16), (False, "ifft", 1, 16), (False, "fft", 1, 20), (False, "ifft", 1, 20),
              (False, "fft", 64, 12), (False, "ifft", 64, 12), (True, "fft", 1, 16))
OPEN_ALL_SHAPES = ((1, 12), (64, 12), (1, 16))
CHAIN_M, CHAIN_LOG_N = 4, 12


def nontrivial_muls(kind, m, log_n):
    n = 1 << log_n
    per_row = log_n * n // 2 - (n - 1) + (n if kind != "fft" else 0)
    return m * per_row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--only", nargs="*", choices=("fft", "open_all", "chain"), default=("fft", "open_all", "chain"))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_point_fft.py needs a CUDA device")
    import bench
    import fr_fft_model as fm
    import bls_model as bm
    import pairing_b200._native as nat
    from pairing_b200.device import DeviceEngine
    eng = DeviceEngine(device=0)
    gpu = {"name": torch.cuda.get_device_name(0)}
    try:
        gpu["nvidia_smi"] = subprocess.check_output(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv"],
                                                    text=True).strip().splitlines()[-1]
    except Exception as e:                                    # noqa: BLE001 -- recorded, not fatal
        gpu["nvidia_smi"] = "unavailable: %s" % e
    pa, qa, _, _ = bench.make_inputs(eng, 1 << 20, 0x9F7, torch, np)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=eng.device)
    gen = torch.Generator(device=eng.device).manual_seed(0x9F8)

    def timed(*fns):
        """medians of the fns, launched alternately after one warm-up each"""
        for fn in fns:
            fn()
        ts = [[] for _ in fns]
        for _ in range(args.reps):
            for k, fn in enumerate(fns):
                flush.fill_(1)
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                fn()
                b.record()
                b.synchronize()
                ts[k].append(a.elapsed_time(b))
        return [sorted(t)[len(t) // 2] for t in ts]

    def rows_of(pts, count, off=0):
        return pts[(torch.arange(count, device=eng.device) + off) % pts.shape[0]].contiguous()

    def fr_of(*shape, bits=60):
        x = torch.randint(-(1 << 63), (1 << 63) - 1, shape + (4,), dtype=torch.int64, device=eng.device, generator=gen)
        x[..., 3] &= (1 << bits) - 1
        return x

    def jacobian(aff, g2):
        """affine rows (no identities) -> Jacobian rows with z = one"""
        w = 12 if g2 else 6
        one = torch.from_numpy(np.array(bm.limbs64(bm.to_mont(1), 6), dtype=np.uint64).view(np.int64)).to(eng.device)
        jac = torch.zeros((aff.shape[0], 3 * w), dtype=torch.int64, device=eng.device)
        jac[:, :2 * w] = aff[:, :2 * w]
        jac[:, 2 * w:2 * w + 6] = one
        return jac

    rows = []
    for g2, kind, m, log_n in FFT_SHAPES if "fft" in args.only else ():
        n = 1 << log_n
        pts = qa if g2 else pa
        x = rows_of(pts, m * n).reshape(m, n, -1).contiguous()
        out = torch.empty_like(x)
        cnt = nontrivial_muls(kind, m, log_n)
        bases = jacobian(rows_of(pts, cnt, 7), g2)
        k = fr_of(cnt, bits=62)
        wout = torch.empty_like(bases)
        fft = eng.g2_fft if g2 else eng.g1_fft
        wnaf = eng.g2_wnaf_mul if g2 else eng.g1_wnaf_mul
        ms_f, ms_w = timed(lambda: fft(x, kind, out=out), lambda: wnaf(bases, k, out=wout))
        rows.append({"call": ("g2" if g2 else "g1") + "_fft", "kind": kind, "m": m, "log_n": log_n, "ms": ms_f, "nontrivial_muls": cnt,
                     "ns_per_mul": ms_f * 1e6 / cnt, "wnaf_ms": ms_w, "wnaf_ns_per_mul": ms_w * 1e6 / cnt, "ratio_to_wnaf": ms_f / ms_w})
        print(json.dumps(rows[-1]), flush=True)
        del x, out, bases, k, wout
        eng._scratch.clear()
        torch.cuda.empty_cache()

    for m, log_n in OPEN_ALL_SHAPES if "open_all" in args.only else ():
        n = 1 << log_n
        table = eng.kzg_open_all_prepare(rows_of(pa, n), log_n)
        p = fr_of(m, n)
        (ms,) = timed(lambda: eng.kzg_open_all(table, p))
        (ms_prep,) = timed(lambda: eng.kzg_open_all_prepare(rows_of(pa, n), log_n, out=table))
        rows.append({"call": "kzg_open_all", "m": m, "log_n": log_n, "ms": ms, "openings": m * n, "us_per_opening": ms * 1e3 / (m * n),
                     "prepare_ms": ms_prep})
        print(json.dumps(rows[-1]), flush=True)
        del table, p
        eng._scratch.clear()
        torch.cuda.empty_cache()

    if "chain" in args.only:
        m, log_n = CHAIN_M, CHAIN_LOG_N
        n = 1 << log_n
        srs = rows_of(pa, n)
        table = eng.kzg_open_all_prepare(srs, log_n)
        p = fr_of(m, n)
        w = fm.fr_root(log_n)
        z = torch.from_numpy(np.array([bm.limbs64(bm.fr_to_mont(pow(w, k, bm.R_ORDER)), 4) for k in range(n)] * m, dtype=np.uint64)
                             .view(np.int64)).to(eng.device)
        prep = p.repeat_interleave(n, dim=0).contiguous()
        res = {}

        def open_all():
            res["all"] = eng.kzg_open_all(table, p)

        def chain():
            res["chain"] = eng.kzg_open(srs[:n - 1], prep, z)

        ms_a, ms_c = timed(open_all, chain)
        ya, pra = res["all"]
        yc, prc = res["chain"]
        agree = bool(torch.equal(ya.reshape(-1, 4), yc) and torch.equal(pra.reshape(-1, nat.W_G1A), prc))
        rows.append({"call": "kzg_open_all_vs_open_chain", "m": m, "log_n": log_n, "openings": m * n, "ms_open_all": ms_a, "ms_chain": ms_c,
                     "speedup": ms_c / ms_a, "outputs_agree": agree})
        print(json.dumps(rows[-1]), flush=True)
    out = {"gpu": gpu, "reps": args.reps, "flush_bytes": 256 << 20,
           "inputs": "bench.make_inputs(eng, 2^20, 0x9F7) points (repeated); coefficients torch.randint limbs, top limb masked to 60 bits; "
                     "wNAF scalars masked to 62 bits",
           "rows": rows}
    with open(args.out, "w") as fh:
        json.dump(out, fh, indent=1)


if __name__ == "__main__":
    main()
