"""KZG commitments on one GPU: bls_kzg_commit_dev, bls_kzg_open_dev, bls_kzg_verify_dev and bls_kzg_verify_rlc_dev (through
DeviceEngine).
Shapes: commit and open at 1 x 2^20, 1 x 2^24 and 64 x 2^14 coefficients; verify at 2^16 and 2^20 proofs; the randomized check
at 2^20 proofs.  Points are bench.make_inputs' 2^20 subgroup points, repeated past 2^20 (the SRS rows, C and the proofs);
coefficients, y, z and rho are torch.randint limbs with the top limb masked to 60 bits (canonical).  The openings do not
verify; the kernels have no early exit, so a verdict of 0 costs what a verdict of 1 costs.
Each call is timed by CUDA events as the median of --reps launches after one warm-up, with a 256 MiB write between launches
(the L2 holds nothing of the previous launch).  verify is timed alternately, in the same process, with the chain of existing
calls that computes the same verdicts: bls_fr_op_dev (r - y and into_repr), bls_g1_msm_batch_dev over [C, g, W] with [1, r - y, z]
(n = 3, in batches of 2^16, its limit), two bls_miller_loop_shared_q_dev on the pvk's prepared points, the Fq12 product
(bls_pair_field_op_dev), bls_final_exponentiation_dev and a comparison with one; the verdicts are compared.  The G1 term
P_j = C_j - y_j g + z_j W_j is timed both ways: the chain's n = 3 multiexp (plus the into-affine copy) against k_kzg_term plus
the normalisation, the latter from a torch.profiler pass.  A profiler pass per shape (one call, after the timed ones) splits
each call's GPU time into the scan, the multiexp and the rest.
    python tools/bench_kzg.py --out kzg.json
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT]

OPEN_SHAPES = ((1, 1 << 20), (1, 1 << 24), (64, 1 << 14))
VERIFY_M = (1 << 16, 1 << 20)
RLC_M = (1 << 20,)
MSM_BATCH_MAX = 1 << 16


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--only", nargs="*", choices=("open", "verify", "rlc"), default=("open", "verify", "rlc"))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_kzg.py needs a CUDA device")
    import bench
    import pairing_b200._native as nat
    from pairing_b200.device import DeviceEngine
    eng = DeviceEngine(device=0)
    ctx = eng.ctx
    gpu = {"name": torch.cuda.get_device_name(0)}
    try:
        gpu["nvidia_smi"] = subprocess.check_output(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv"],
                                                    text=True).strip().splitlines()[-1]
    except Exception as e:                                    # noqa: BLE001 -- recorded, not fatal
        gpu["nvidia_smi"] = "unavailable: %s" % e
    pa, qa, _, _ = bench.make_inputs(eng, 1 << 20, 0x3A5E, torch, np)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=eng.device)
    gen = torch.Generator(device=eng.device).manual_seed(0x6A2E)
    stream = eng._stream()

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

    def profile(fn):
        """GPU time of one call by kernel group: {"scan", "msm", "term", "rest"} ms and {kernel: ms}"""
        flush.fill_(1)
        torch.cuda.synchronize()
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        groups = {"scan": 0.0, "msm": 0.0, "term": 0.0, "rest": 0.0}
        kern = {}
        for ev in prof.key_averages():
            if ev.self_device_time_total <= 0 or "fill" in ev.key.lower() or "memcpy" in ev.key.lower() or "memset" in ev.key.lower():
                continue
            ms = ev.self_device_time_total / 1e3
            kern[ev.key[:60]] = kern.get(ev.key[:60], 0.0) + ms
            g = "scan" if "k_kzg_scan" in ev.key else "msm" if "msm" in ev.key else \
                "term" if ("k_kzg_term" in ev.key or "batch_normalization" in ev.key) else "rest"
            groups[g] += ms
        return groups, kern

    def rows_of(pts, count, off):
        return pts[(torch.arange(count, device=eng.device) + off) % pts.shape[0]].contiguous()

    def fr_of(*shape):
        x = torch.randint(-(1 << 63), (1 << 63) - 1, shape + (4,), dtype=torch.int64, device=eng.device, generator=gen)
        x[..., 3] &= (1 << 60) - 1                            # canonical: < 2^252 < r
        return x

    host = lambda t: t.cpu().numpy().view(np.uint64)  # noqa: E731
    rows = []
    for m, n in OPEN_SHAPES if "open" in args.only else ():
        srs = rows_of(pa, n, 0)
        p = fr_of(m, n)
        z = fr_of(m)
        c = torch.empty((m, nat.W_G1A), dtype=torch.int64, device=eng.device)
        ms_c, ms_o = timed(lambda: eng.kzg_commit(srs, p, out=c), lambda: eng.kzg_open(srs, p, z))
        g_o, k_o = profile(lambda: eng.kzg_open(srs, p, z))
        g_c, _ = profile(lambda: eng.kzg_commit(srs, p, out=c))
        rows.append({"call": "commit+open", "m": m, "n": n, "ms_commit": ms_c, "ms_open": ms_o, "gpu_ms_open": g_o, "gpu_ms_commit": g_c,
                     "scan_share_of_open_gpu_time": g_o["scan"] / sum(g_o.values()), "gpu_ms_open_kernels": k_o})
        print(json.dumps(rows[-1]), flush=True)
        del srs, p, z, c
        eng._scratch.clear()
        torch.cuda.empty_cache()

    g_row, h_rows = host(pa[:1])[0], host(qa[:2])
    pvk = eng.kzg_prepare_verifying_key(g_row, h_rows[0], h_rows[1])
    off = {name: getattr(nat.KzgPvkC, name).offset // 8 for name in ("h_prepared", "neg_tau_h_prepared", "g", "h")}
    inf = DeviceEngine.jacobian_to_affine_rows(torch.zeros((1, nat.W_G1), dtype=torch.int64, device=eng.device), 6)
    one = eng.pairing(inf, qa[:1])[0]                         # e(infinity, Q) = one
    for m in VERIFY_M if "verify" in args.only else ():
        cc, w = rows_of(pa, m, 100), rows_of(pa, m, 300)
        y, z = fr_of(m), fr_of(m)
        out = torch.empty(m, dtype=torch.uint8, device=eng.device)
        # the chain's buffers
        gs = pvk[off["g"]:off["g"] + nat.W_G1A][None].expand(m, nat.W_G1A)
        bases = torch.stack([cc, gs, w], dim=1).contiguous()
        scal = torch.zeros((m, 3, 4), dtype=torch.int64, device=eng.device)
        scal[:, 0, 0] = 1
        ny, zr = torch.empty_like(y), torch.empty_like(z)
        pt = torch.empty((m, nat.W_G1), dtype=torch.int64, device=eng.device)
        ml = [torch.empty((m, nat.W_FQ12), dtype=torch.int64, device=eng.device) for _ in range(2)]
        fe = torch.empty((m, nat.W_FQ12), dtype=torch.int64, device=eng.device)
        chain_ok = torch.empty(m, dtype=torch.bool, device=eng.device)

        def verify():
            eng.kzg_verify(pvk, cc, y, z, w, out=out)

        def term_chain():
            eng.fr_op("neg", y, out=ny)
            eng.fr_op("into_repr", ny, out=ny)
            eng.fr_op("into_repr", z, out=zr)
            scal[:, 1] = ny
            scal[:, 2] = zr
            for s in range(0, m, MSM_BATCH_MAX):
                e = min(m, s + MSM_BATCH_MAX)
                eng.msm_batch(bases[s:e], scal[s:e], out=pt[s:e])
            return DeviceEngine.jacobian_to_affine_rows(pt, 6)

        def chain():
            pt_aff = term_chain()
            ctx.call_dev("bls_miller_loop_shared_q_dev", pt_aff.data_ptr(), pvk.data_ptr() + 8 * off["h_prepared"], ml[0].data_ptr(), m, 0, stream)
            ctx.call_dev("bls_miller_loop_shared_q_dev", w.data_ptr(), pvk.data_ptr() + 8 * off["neg_tau_h_prepared"], ml[1].data_ptr(), m, 0, stream)
            ctx.call_dev("bls_pair_field_op_dev", 12, nat.OPS["mul"], ml[0].data_ptr(), ml[1].data_ptr(), ml[0].data_ptr(), None, m, stream)
            _, some = eng.final_exponentiation(ml[0], out=fe)
            torch.logical_and((fe == one[None]).all(dim=1), some.bool(), out=chain_ok)

        groups, kern = profile(verify)
        ms_v, ms_c, ms_t = timed(verify, chain, term_chain)
        verify(); chain()
        agree = bool(torch.equal(out.bool(), chain_ok))
        rows.append({"call": "verify", "m": m, "ms": ms_v, "ms_chain": ms_c, "speedup_vs_chain": ms_c / ms_v, "proofs_per_s": m / ms_v * 1e3,
                     "g1_term_joint_gpu_ms": groups["term"], "g1_term_msm_n3_ms": ms_t, "gpu_ms": groups, "gpu_ms_kernels": kern,
                     "verdicts_agree_with_chain": agree, "verdicts_true": int(out.sum().item())})
        print(json.dumps(rows[-1]), flush=True)
        del cc, w, y, z, out, bases, scal, ny, zr, pt, ml, fe, chain_ok
        eng._scratch.clear()
        torch.cuda.empty_cache()
    for m in RLC_M if "rlc" in args.only else ():
        cc, w = rows_of(pa, m, 100), rows_of(pa, m, 300)
        y, z, rho = fr_of(m), fr_of(m), fr_of(m)
        out1 = torch.zeros(1, dtype=torch.uint8, device=eng.device)

        def rlc():
            eng.kzg_verify_rlc(pvk, cc, y, z, w, rho, out=out1)

        (ms_r,) = timed(rlc)
        groups, kern = profile(rlc)
        rows.append({"call": "verify_rlc", "m": m, "ms": ms_r, "proofs_per_s": m / ms_r * 1e3, "gpu_ms": groups, "gpu_ms_kernels": kern,
                     "verdict": int(out1.item())})
        print(json.dumps(rows[-1]), flush=True)
    res = {"gpu": gpu, "reps": args.reps, "flush_bytes": 256 << 20,
           "inputs": "bench.make_inputs(eng, 2^20, 0x3A5E) points for the SRS, C, W and the key (repeated past 2^20); coefficients, y, "
                     "z and rho torch.randint limbs, top limb masked to 60 bits (canonical)",
           "rows": rows}
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
