"""Multi-scalar multiplication (bls_g1_msm_dev / bls_g2_msm_dev) against the per-point wNAF batch over the same points and
scalars, on one GPU.

For every size n: the library's window (window = 0) and a sweep of the bucket width c, each timed by CUDA events as the
median of --reps launches after one warm-up, with a 256 MiB write between launches (as bench.py does) so that no launch
finds its inputs in L2; then g*_wnaf_mul_dev over the same points and scalars, alternating with the MSM launches.

Work counted (algorithmic MAC32, M = 300 per Fq product): one mixed addition per non-zero signed digit, 2 * 2^(c-1)
additions per window for the bucket reduction, (W - 1) * c doublings + W additions for the Horner step (W = ceil(257 / c));
G1 11 / 16 / 7 M per mixed addition / addition / doubling, G2 29 / 43 / 16 M.  The segment tree of the reduction
(log2 of the segment count rounds) is not counted.  Share of peak = that work over the time, divided by the IMAD.WIDE
rate measured in the same run (bls_imad_peak variant 0).

    python tools/bench_msm.py --out msm.json

--batch: batched MSM (bls_g*_msm_batch_dev), G1 and G2, shared and separate bases, at the (m, n) shapes of BATCH_SHAPES.
Per shape: the library's window and a sweep of c, each the median of --reps launches as above; then the batch alternating with
ONE bls_g*_msm_dev call at n (the single sum, times m, is what a loop of m calls costs).  Work as above, per sum.

    python tools/bench_msm.py --batch --out msm_batch.json
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT]

M = 300
MONT_ONE = [0x760900000002fffd, 0xebf4000bc40c0002, 0x5f48985753c758ba, 0x77ce585370525745, 0x5c071a97a256ec6d, 0x15f65ec3fa80e493]   # fq.rs:22-30
COST = {False: (11, 16, 7), True: (29, 43, 16)}     # Fq products per mixed addition, addition, doubling
BATCH_SHAPES = [(1, 1 << 12), (16, 1 << 12), (64, 1 << 12), (256, 1 << 12), (1024, 1 << 10), (64, 1 << 16), (4, 1 << 20)]
BATCH_G1_ONLY = {(4, 1 << 20)}


def nonzero_digits(k, c, np):
    """(n,) count of non-zero signed c-bit digits per scalar, the recoding of kernels_msm.cu (digits in (-2^(c-1), 2^(c-1)])"""
    n = k.shape[0]
    nwin = (257 + c - 1) // c
    mask, half = np.uint64((1 << c) - 1), np.uint64(1 << (c - 1))
    carry = np.zeros(n, dtype=np.uint64)
    count = np.zeros(n, dtype=np.int64)
    for j in range(nwin):
        bit = c * j
        raw = np.zeros(n, dtype=np.uint64)
        if bit < 256:
            w, o = bit // 64, bit % 64
            raw = k[:, w] >> np.uint64(o)
            if o and w < 3:
                raw |= k[:, w + 1] << np.uint64(64 - o)
            raw &= mask
        d = raw + carry
        carry = (d > half).astype(np.uint64)
        count += (d != 0) & (d != (mask + np.uint64(1)))
    return count


def macs(g2, entries, n_windows_c):
    nwin, c = n_windows_c
    madd, add, dbl = COST[g2]
    return M * (madd * entries + add * (2 * nwin * (1 << (c - 1)) + nwin) + dbl * c * (nwin - 1))


def library_window(n, m):
    """the c of window = 0 (msm_default_window in kernels_msm.cu)"""
    lg = max(n.bit_length() - 1, 0)
    c = min(20, max(7 if m > 1 and lg <= 10 else 8, lg - 5))
    while ((257 + c - 1) // c) * m * n >= 1 << 31:
        c += 1
    return c


def batch_macs(g2, entries, m, c):
    """work of m sums with `entries` non-zero digits in all: the accumulation, and the reduction and Horner step per sum"""
    nwin = (257 + c - 1) // c
    return macs(g2, entries, (nwin, c)) + (m - 1) * macs(g2, 0, (nwin, c))


def run_batch(args, eng, peak, pa, qa, k, once, median, timed, np, torch):
    """the --batch mode: (summary, rows)"""
    import pairing_b200._native as nat
    k_host = k.cpu().numpy().view(np.uint64)
    rows, summary = [], []
    for g2 in (False, True):
        group = "G2" if g2 else "G1"
        bases_all = qa if g2 else pa
        for m, n in BATCH_SHAPES:
            if g2 and (m, n) in BATCH_G1_ONLY:
                continue
            lg = n.bit_length() - 1
            kk = k[:m * n].reshape(m, n, 4)
            entries = {}
            for shared in (True, False):
                mode = "shared" if shared else "separate"
                b = bases_all[:n] if shared else bases_all[:m * n].reshape(m, n, -1)
                out = torch.empty((m, nat.W_G2 if g2 else nat.W_G1), dtype=torch.int64, device=eng.device)
                one = out[:1].clone()
                batch = lambda c: eng.msm_batch(b, kk, g2=g2, window=c, out=out)
                single = lambda: eng.msm(bases_all[:n], k[:n], g2=g2, out=one)
                batch(0)
                ref = out.clone()
                sweep = {}
                for c in sorted({library_window(n, m)} | set(range(max(5, lg - 6), min(20, lg + 1) + 1))):
                    try:
                        eng.ctx.msm_batch_scratch_bytes(2 if g2 else 1, n, m, c)
                    except ValueError:
                        continue                                  # outside the limits of one call
                    sweep[c] = timed(lambda: batch(c))
                    assert torch.equal(out, ref), "window %d changes the result" % c
                    if c not in entries:
                        entries[c] = int(nonzero_digits(k_host[:m * n], c, np).sum())
                    w = batch_macs(g2, entries[c], m, c)
                    rows.append({"group": group, "m": m, "n": n, "bases": mode, "window": c, "ms": sweep[c], "mac32": w,
                                 "share_of_imad_peak": w / (sweep[c] * 1e-3) / peak})
                single()
                b_ms, s_ms = [], []
                for _ in range(args.reps):                        # the batch and one single MSM at n alternate
                    b_ms.append(once(lambda: batch(0)))
                    s_ms.append(once(single))
                bt, st = median(b_ms), median(s_ms)
                c0 = library_window(n, m)
                best = min(sweep, key=sweep.get)
                summary.append({"group": group, "m": m, "n": n, "bases": mode, "batch_ms": bt, "single_ms": st, "loop_ms": m * st,
                                "speedup": m * st / bt, "sums_per_s": m / (bt * 1e-3), "window": c0,
                                "share_of_imad_peak": batch_macs(g2, entries[c0], m, c0) / (bt * 1e-3) / peak,
                                "best_window": best, "best_ms": sweep[best], "library_over_best": sweep[c0] / sweep[best]})
                print(json.dumps(summary[-1]), flush=True)
    return summary, rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--g1-max", type=int, default=24)
    ap.add_argument("--g2-max", type=int, default=22)
    ap.add_argument("--min", type=int, default=10)
    ap.add_argument("--step", type=int, default=2)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--seed", type=int, default=0x5DBE62598D313D76)
    ap.add_argument("--batch", action="store_true", help="batched MSM at BATCH_SHAPES instead of the single-sum sweep")
    args = ap.parse_args()

    import numpy as np
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_msm.py needs a CUDA device")
    import bench
    from pairing_b200.device import DeviceEngine
    import pairing_b200._native as nat

    eng = DeviceEngine(device=0)
    ctx = eng.ctx
    gpu = {"name": torch.cuda.get_device_name(0)}
    try:
        gpu["nvidia_smi"] = subprocess.check_output(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv"],
                                                    text=True).strip().splitlines()[-1]
    except Exception as e:                                    # noqa: BLE001 -- recorded, not fatal
        gpu["nvidia_smi"] = "unavailable: %s" % e
    peak, _ = ctx.imad_peak(0)

    nmax = max(m * n for m, n in BATCH_SHAPES) if args.batch else 1 << max(args.g1_max, args.g2_max)
    pa, qa, p_jac, k = bench.make_inputs(eng, nmax, args.seed, torch, np)
    one = torch.tensor(np.array(MONT_ONE, dtype=np.uint64).view(np.int64), device=eng.device)
    q_jac = torch.zeros((nmax, nat.W_G2), dtype=torch.int64, device=eng.device)
    q_jac[:, :24] = qa[:, :24]
    q_jac[:, 24:30] = one
    k_host = k.cpu().numpy().view(np.uint64)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=eng.device)
    torch.cuda.synchronize()

    def once(fn):
        flush.fill_(1)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        return a.elapsed_time(b)

    def median(ts):
        return sorted(ts)[len(ts) // 2]

    def timed(fn):
        fn()
        return median([once(fn) for _ in range(args.reps)])

    if args.batch:
        summary, rows = run_batch(args, eng, peak, pa, qa, k, once, median, timed, np, torch)
        res = {"gpu": gpu, "imad_peak_mac32_per_s": peak, "reps": args.reps, "flush_bytes": 256 << 20,
               "scalars": "bench.make_inputs scalars (SplitMix64, < 2^254): sum j takes scalars j n .. j n + n - 1; bases = bench.make_inputs "
                          "points, the first n (shared) or the first m n (separate)", "summary": summary, "rows": rows}
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
        return

    digit_cache = {}

    def entries(c, n):
        if c not in digit_cache:
            digit_cache[c] = np.concatenate([[0], np.cumsum(nonzero_digits(k_host, c, np))])
        return int(digit_cache[c][n])

    rows, summary = [], []
    for g2, lgmax in ((False, args.g1_max), (True, args.g2_max)):
        bases_aff, bases_jac = (qa, q_jac) if g2 else (pa, p_jac)
        for lg in range(args.min, lgmax + 1, args.step):
            n = 1 << lg
            b, kk, bj = bases_aff[:n], k[:n], bases_jac[:n]
            out = torch.empty((1, nat.W_G2 if g2 else nat.W_G1), dtype=torch.int64, device=eng.device)
            wout = torch.empty_like(bj)
            msm = lambda c: eng.msm(b, kk, g2=g2, window=c, out=out)
            wnaf = (lambda: eng.g2_wnaf_mul(bj, kk, out=wout)) if g2 else (lambda: eng.g1_wnaf_mul(bj, kk, out=wout))
            msm(0)
            ref = out.clone()
            sweep = {}
            for c in range(max(3, lg - 9), min(20, lg + 1) + 1):
                sweep[c] = timed(lambda: msm(c))
                assert torch.equal(out, ref), "window %d changes the result" % c
                nwin = (257 + c - 1) // c
                w = macs(g2, entries(c, n), (nwin, c))
                rows.append({"group": "G2" if g2 else "G1", "n": n, "window": c, "ms": sweep[c], "mac32": w,
                             "share_of_imad_peak": w / (sweep[c] * 1e-3) / peak})
            wnaf()
            h_ms, w_ms = [], []
            for _ in range(args.reps):                            # the MSM and the wNAF batch alternate
                h_ms.append(once(lambda: msm(0)))
                w_ms.append(once(wnaf))
            h, wn = median(h_ms), median(w_ms)
            best = min(sweep, key=sweep.get)
            summary.append({"group": "G2" if g2 else "G1", "n": n, "heuristic_ms": h, "best_window": best, "best_ms": sweep[best],
                            "heuristic_over_best": h / sweep[best], "wnaf_batch_ms": wn, "wnaf_over_msm": wn / h})
            print(json.dumps(summary[-1]), flush=True)
    res = {"gpu": gpu, "imad_peak_mac32_per_s": peak, "reps": args.reps, "flush_bytes": 256 << 20,
           "scalars": "bench.make_inputs scalars (SplitMix64, < 2^254), bases = bench.make_inputs points", "summary": summary, "rows": rows}
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
