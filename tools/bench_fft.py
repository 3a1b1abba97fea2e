"""Radix-2 FFT over Fr (bls_fr_fft_dev through DeviceEngine.fr_fft) on one GPU.
Shapes: every kind at log_n = 10, 12, 16, 20, 24, 26 with m = 1; the Groth16 shape m = 3 at 2^20; m = 256 at 2^10.
Each shape is timed by CUDA events as the median of --reps launches after one warm-up, out of place, with a 256 MiB write
between launches (as bench.py does) so that no launch finds its inputs in L2.
Work counted (algorithmic MAC32): (n / 2) * log_n butterflies per polynomial, one Fr product of 128 MAC32 each (fr.cuh);
the inter-pass twiddles, the coset and n^-1 scalings and the table set-up are not counted.  Share of peak = that work over
the time, divided by the IMAD.WIDE rate measured in the same run (bls_imad_peak variant 0).  HBM share = one read and one
write of m * n * 32 bytes per pass over the time, divided by 7.7 TB/s.
    python tools/bench_fft.py --out fft.json
--groth16-h times Groth16's quotient polynomial instead (bls_fr_groth16_h_dev through DeviceEngine.groth16_h) for m proofs
of len = n evaluations, m = 1 at n = 2^16, 2^20, 2^22, 2^24, m = 64 at 2^12 and m = 8 at 2^20, under the same conditions.
Each shape also times, in the same process, the fr_fft calls the one call contains: ifft and coset_fft of 3m polynomials
and icoset_fft of m, in place.
    python tools/bench_fft.py --groth16-h --out groth16_h.json
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT]

MAC_PER_PRODUCT = 128
HBM_BYTES_PER_S = 7.7e12
KINDS = ["fft", "ifft", "coset_fft", "icoset_fft"]


def passes(log_n):
    """passes of kernels_fft.cu: one up to 2^10, else ceil(log_n / 10)"""
    return 1 if log_n <= 10 else (log_n + 9) // 10


def bench_groth16_h(eng, timed, gen):
    import torch
    rows = []
    for lg, m in ((16, 1), (20, 1), (22, 1), (24, 1), (12, 64), (20, 8)):
        n = 1 << lg
        abc = torch.randint(-(1 << 63), (1 << 63) - 1, (3 * m, n, 4), dtype=torch.int64, device=eng.device, generator=gen)
        abc[..., 3] &= (1 << 60) - 1
        a, b, c = (abc[i * m:(i + 1) * m].clone() for i in range(3))
        out = torch.empty((m, n - 1, 4), dtype=torch.int64, device=eng.device)

        def transforms():
            eng.fr_fft(abc, "ifft", out=abc)
            eng.fr_fft(abc, "coset_fft", out=abc)
            eng.fr_fft(abc[:m], "icoset_fft", out=abc[:m])

        ms_call = timed(lambda: eng.groth16_h(a, b, c, out=out))
        ms_fft = timed(transforms)
        rows.append({"log_n": lg, "m": m, "passes": passes(lg), "ms_groth16_h": ms_call, "ms_fft_calls": ms_fft,
                     "ratio": ms_call / ms_fft, "ms_per_proof": ms_call / m})
        print(json.dumps(rows[-1]), flush=True)
        del abc, a, b, c, out
        eng._scratch.clear()
        torch.cuda.empty_cache()
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--sizes", default="10,12,16,20,24,26")
    ap.add_argument("--groth16-h", action="store_true", help="time Groth16's quotient polynomial H instead of the transforms")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_fft.py needs a CUDA device")
    from pairing_b200.device import DeviceEngine
    eng = DeviceEngine(device=0)
    gpu = {"name": torch.cuda.get_device_name(0)}
    try:
        gpu["nvidia_smi"] = subprocess.check_output(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv"],
                                                    text=True).strip().splitlines()[-1]
    except Exception as e:                                    # noqa: BLE001 -- recorded, not fatal
        gpu["nvidia_smi"] = "unavailable: %s" % e
    peak, _ = eng.ctx.imad_peak(0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=eng.device)
    gen = torch.Generator(device=eng.device).manual_seed(0x5EED)

    def median(ts):
        return sorted(ts)[len(ts) // 2]

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
        return median(ts)

    if args.groth16_h:
        res = {"gpu": gpu, "reps": args.reps, "flush_bytes": 256 << 20,
               "inputs": "torch.randint limbs, top limb masked to 60 bits (canonical), len = n evaluations per proof",
               "rows": bench_groth16_h(eng, timed, gen)}
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
        return
    shapes = [(kind, lg, 1) for lg in (int(x) for x in args.sizes.split(",")) for kind in KINDS]
    shapes += [(kind, 20, 3) for kind in KINDS] + [(kind, 10, 256) for kind in KINDS]
    rows = []
    for kind, lg, m in shapes:
        n = 1 << lg
        a = torch.randint(-(1 << 63), (1 << 63) - 1, (m, n, 4), dtype=torch.int64, device=eng.device, generator=gen)
        a[..., 3] &= (1 << 60) - 1                            # canonical: < 2^252 < r
        out = torch.empty_like(a)
        ms = timed(lambda: eng.fr_fft(a, kind, out=out))
        mac = m * (n // 2) * lg * MAC_PER_PRODUCT
        hbm = 2 * passes(lg) * m * n * 32
        rows.append({"kind": kind, "log_n": lg, "m": m, "passes": passes(lg), "ms": ms, "mac32": mac,
                     "share_of_imad_peak": mac / (ms * 1e-3) / peak, "hbm_bytes": hbm,
                     "share_of_hbm": hbm / (ms * 1e-3) / HBM_BYTES_PER_S})
        print(json.dumps(rows[-1]), flush=True)
        del a, out
        torch.cuda.empty_cache()
    res = {"gpu": gpu, "imad_peak_mac32_per_s": peak, "reps": args.reps, "flush_bytes": 256 << 20,
           "inputs": "torch.randint limbs, top limb masked to 60 bits (canonical)", "rows": rows}
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
