"""Groth16 verification on one GPU: bls_groth16_verify_dev (DeviceEngine.groth16_verify) and the randomized check
bls_groth16_verify_rlc_dev (DeviceEngine.groth16_verify_rlc).
Shapes: per-proof verification at m = 1, 64, 2^12 and 2^16; the randomized check at m = 64, 2^12, 2^16 and 2^20; each with
num_inputs = 1 and 64.  Points are bench.make_inputs' 2^20 subgroup points (repeated past 2^20): the vk points, ic, and the
proofs' A, B, C.  The proofs do not verify; the kernels have no early exit, so a verdict of 0 costs what a verdict of 1 costs.
Each call is timed by CUDA events as the median of --reps launches after one warm-up, with a 256 MiB write between launches
(the L2 holds nothing of the previous launch).  In the same process, alternated with the fused call, the script times the
chain of existing calls that computes the same verdicts: into_repr of the inputs (bls_fr_op_dev), bls_g1_msm_batch_dev,
bls_miller_loop_dev(A, B), bls_miller_loop_shared_q_dev for (acc, -gamma) and (C, -delta) on the prepared points of the pvk,
two Fq12 products (bls_pair_field_op_dev), bls_final_exponentiation_dev and a comparison; its verdicts are checked against the
fused call's.  A torch.profiler pass per shape (one call, after the timed ones) records each kernel's GPU time and splits the call's
into the msm kernels and the rest.
    python tools/bench_groth16_verify.py --out groth16_verify.json
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT]

VERIFY_M = (1, 64, 1 << 12, 1 << 16)
RLC_M = (64, 1 << 12, 1 << 16, 1 << 20)
NUM_INPUTS = (1, 64)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=7)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_groth16_verify.py needs a CUDA device")
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
    gen = torch.Generator(device=eng.device).manual_seed(0x6017)

    def timed_pair(f1, f2):
        """medians of f1 and f2, launched alternately after one warm-up each"""
        f1(); f2()
        ts = ([], [])
        for _ in range(args.reps):
            for k, fn in enumerate((f1, f2)):
                flush.fill_(1)
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                fn()
                b.record()
                b.synchronize()
                ts[k].append(a.elapsed_time(b))
        return [sorted(t)[len(t) // 2] for t in ts]

    def profile(fn):
        """GPU time of one call: (msm kernels, the other kernels, {kernel: ms}), ms"""
        flush.fill_(1)
        torch.cuda.synchronize()
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        msm = rest = 0.0
        kern = {}
        for ev in prof.key_averages():
            if ev.self_device_time_total <= 0 or "fill" in ev.key.lower() or "memcpy" in ev.key.lower() or "memset" in ev.key.lower():
                continue
            ms = ev.self_device_time_total / 1e3
            kern[ev.key[:60]] = kern.get(ev.key[:60], 0.0) + ms
            if "msm" in ev.key:
                msm += ms
            else:
                rest += ms
        return msm, rest, kern

    def rows_of(pts, count, off):
        return pts[(torch.arange(count, device=eng.device) + off) % pts.shape[0]].contiguous()

    def inputs_of(m, ni):
        x = torch.randint(-(1 << 63), (1 << 63) - 1, (m, ni, 4), dtype=torch.int64, device=eng.device, generator=gen)
        x[..., 3] &= (1 << 60) - 1                            # canonical: < 2^252 < r
        return x

    host = lambda t: t.cpu().numpy().view(np.uint64)  # noqa: E731
    pvk_np = ctx.groth16_prepare_verifying_key(host(pa[:1])[0], *host(qa[:3]))
    pvk = torch.from_numpy(pvk_np.view(np.int64)).to(eng.device)
    f = {name: getattr(nat.Groth16PvkC, name).offset // 8 for name in ("neg_gamma_g2", "neg_delta_g2", "alpha_g1_beta_g2", "neg_gamma_g2_affine")}
    ab = pvk[f["alpha_g1_beta_g2"]:f["alpha_g1_beta_g2"] + nat.W_FQ12]
    stream = eng._stream()
    rows = []
    for ni in NUM_INPUTS:
        ic = rows_of(pa, ni + 1, 3)
        for m in VERIFY_M:
            proofs = torch.cat([rows_of(pa, m, 100), rows_of(qa, m, 200), rows_of(pa, m, 300)], dim=1).contiguous()
            inputs = inputs_of(m, ni)
            out = torch.empty(m, dtype=torch.uint8, device=eng.device)
            # the chain's buffers
            one = torch.zeros((m, 1, 4), dtype=torch.int64, device=eng.device)
            one[..., 0] = 1
            reprs = torch.empty_like(inputs)
            scal = torch.empty((m, ni + 1, 4), dtype=torch.int64, device=eng.device)
            acc = torch.empty((m, nat.W_G1), dtype=torch.int64, device=eng.device)
            ml = [torch.empty((m, nat.W_FQ12), dtype=torch.int64, device=eng.device) for _ in range(3)]
            fe = torch.empty((m, nat.W_FQ12), dtype=torch.int64, device=eng.device)
            chain_ok = torch.empty(m, dtype=torch.bool, device=eng.device)
            a_rows, b_rows, c_rows = proofs[:, :13].contiguous(), proofs[:, 13:38].contiguous(), proofs[:, 38:].contiguous()

            def verify():
                eng.groth16_verify(pvk, ic, proofs, inputs, out=out)

            def chain():
                if ni:
                    eng.fr_op("into_repr", inputs.view(-1, 4), out=reprs.view(-1, 4))
                torch.cat([one, reprs], dim=1, out=scal)
                eng.msm_batch(ic, scal, out=acc)
                acc_aff = DeviceEngine.jacobian_to_affine_rows(acc, 6)
                eng.miller_loop_batch(a_rows, b_rows, out=ml[0])
                ctx.call_dev("bls_miller_loop_shared_q_dev", acc_aff.data_ptr(), pvk.data_ptr() + 8 * f["neg_gamma_g2"], ml[1].data_ptr(), m, 0, stream)
                ctx.call_dev("bls_miller_loop_shared_q_dev", c_rows.data_ptr(), pvk.data_ptr() + 8 * f["neg_delta_g2"], ml[2].data_ptr(), m, 0, stream)
                ctx.call_dev("bls_pair_field_op_dev", 12, nat.OPS["mul"], ml[0].data_ptr(), ml[1].data_ptr(), ml[0].data_ptr(), None, m, stream)
                ctx.call_dev("bls_pair_field_op_dev", 12, nat.OPS["mul"], ml[0].data_ptr(), ml[2].data_ptr(), ml[0].data_ptr(), None, m, stream)
                _, some = eng.final_exponentiation(ml[0], out=fe)
                torch.logical_and((fe == ab[None]).all(dim=1), some.bool(), out=chain_ok)

            ms_v, ms_c = timed_pair(verify, chain)
            verify(); chain()
            agree = bool(torch.equal(out.bool(), chain_ok))
            msm, rest, kern = profile(verify)
            rows.append({"call": "verify", "m": m, "num_inputs": ni, "ms": ms_v, "ms_chain": ms_c, "speedup_vs_chain": ms_c / ms_v,
                         "proofs_per_s": m / ms_v * 1e3, "gpu_ms_msm": msm, "gpu_ms_rest": rest, "gpu_ms_kernels": kern,
                         "verdicts_agree_with_chain": agree, "verdicts_true": int(out.sum().item())})
            print(json.dumps(rows[-1]), flush=True)
            del proofs, inputs, out, one, reprs, scal, acc, ml, fe, chain_ok, a_rows, b_rows, c_rows
        for m in RLC_M:
            proofs = torch.cat([rows_of(pa, m, 100), rows_of(qa, m, 200), rows_of(pa, m, 300)], dim=1).contiguous()
            inputs = inputs_of(m, ni)
            rho = inputs_of(m, 1).view(m, 4).contiguous()
            out1 = torch.zeros(1, dtype=torch.uint8, device=eng.device)

            def rlc():
                eng.groth16_verify_rlc(pvk, ic, proofs, inputs, rho, out=out1)

            ms_r, _ = timed_pair(rlc, lambda: None)
            msm, rest, kern = profile(rlc)
            rows.append({"call": "verify_rlc", "m": m, "num_inputs": ni, "ms": ms_r, "proofs_per_s": m / ms_r * 1e3, "gpu_ms_msm": msm,
                         "gpu_ms_rest": rest, "gpu_ms_kernels": kern, "verdict": int(out1.item())})
            print(json.dumps(rows[-1]), flush=True)
            del proofs, inputs, rho, out1
            eng._scratch.clear()
            torch.cuda.empty_cache()
    res = {"gpu": gpu, "reps": args.reps, "flush_bytes": 256 << 20,
           "inputs": "bench.make_inputs(eng, 2^20, 0x3A5E) points for the vk, ic and the proofs (repeated past 2^20); inputs and rho "
                     "torch.randint limbs, top limb masked to 60 bits (canonical)",
           "rows": rows}
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
