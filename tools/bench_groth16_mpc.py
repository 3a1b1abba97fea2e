"""Times phase 2 of the Groth16 ceremony on one GPU (DeviceEngine.groth16_mpc_new / _contribute / _verify) and writes
--out (JSON) and --md (the table of profiles/groth16_mpc.md).

- mpc_new at 2^16 and 2^20 constraints on tools/bench_groth16_setup.py's circuit(), with its random coefficients and with
  +-1 / +-2^k coefficients, alternated with one bls_g1_wnaf_mul_dev + bls_g2_wnaf_mul_dev batch of as many random 255-bit
  multiplications as the call has G1 and G2 terms; then one profiled call split by kernel.
- contribute with h_len + l_len = 2^21 rows, alternated with bls_g1_wnaf_mul_dev over the same bases with the scalar
  replicated (the comparison that removed a dedicated one-scalar kernel: DESIGN.md).
- verify at 2^20 rows per query with k = 8 contributions, split by the profiler into multiexps and pairings.
Each time is the median of --reps calls after a warm-up, with 256 MiB written between calls; the card, its power limit and
its max SM clock are read in the same process."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tools")]

from bench_groth16_setup import circuit  # noqa: E402


def small_coefficients(abc, seed):
    """the same circuit with every coefficient +-1 or +-2^k (Montgomery form of the canonical values)"""
    import bls_model as bm
    rng = np.random.default_rng(seed)
    vals = [1, bm.R_ORDER - 1] + [(1 << k) for k in range(1, 64)] + [bm.R_ORDER - (1 << k) for k in range(1, 64)]
    table = np.array([bm.limbs64(bm.fr_to_mont(v), 4) for v in vals], dtype=np.uint64)
    return [(off, cons, table[rng.integers(0, len(vals), len(cons))]) for off, cons, _ in abc]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--md", required=True)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--logs", default="16,20")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_groth16_mpc.py needs a CUDA device")
    import oracle_lib as o
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
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=eng.device)
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a).view(np.int64 if a.dtype == np.uint64 else np.int32)).to(eng.device)  # noqa: E731
    g1, g2 = o.generators()
    rng = np.random.default_rng(0x3C)

    def rand_scalars(n):
        k = rng.integers(0, 2 ** 63, size=(n, 4), dtype=np.int64).astype(np.uint64)
        k[:, 3] &= (1 << 62) - 1
        return k

    def points(g2_, n):
        """n random subgroup points: (Jacobian CUDA tensor, affine CUDA tensor)"""
        base = np.repeat(o.g2_from_affine(g2) if g2_ else o.g1_from_affine(g1), n, 0)
        jac = ctx.g2_wnaf_mul(base, rand_scalars(n)) if g2_ else ctx.g1_wnaf_mul(base, rand_scalars(n))
        aff = ctx.g2_into_affine(jac) if g2_ else ctx.g1_into_affine(jac)
        return dev(jac), dev(aff)

    def timed(fns, reps):
        for fn in fns:
            fn()
        ts = [[] for _ in fns]
        for _ in range(reps):
            for i, fn in enumerate(fns):                      # alternated, so both see the same machine state
                flush.fill_(1)
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                fn()
                b.record()
                b.synchronize()
                ts[i].append(a.elapsed_time(b))
        return [sorted(t)[len(t) // 2] for t in ts]

    def split(fn, groups):
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        out = {g: 0.0 for g in groups}
        out["other"] = 0.0
        for ev in prof.key_averages():
            t = ev.self_device_time_total / 1000.0
            if t <= 0:
                continue
            g = next((g for g, keys in groups.items() if any(k in ev.key for k in keys)), "other")
            out[g] += t
        return {k: round(v, 3) for k, v in out.items()}

    res = {"gpu": gpu, "reps": args.reps, "flush_bytes": 256 << 20, "mpc_new": [], "contribute": None, "verify": None}
    pool = 1 << 20
    j1, a1 = points(False, pool)
    j2, a2 = points(True, pool)
    gg1, gg2 = g1[0], g2[0]
    for log_c in [int(x) for x in args.logs.split(",")]:
        n = 1 << log_c
        abc0, na = circuit(log_c, 4, log_c)
        for kind, abc in (("random", abc0), ("small", small_coefficients(abc0, log_c))):
            dabc = [(dev(off), dev(c), dev(k)) for off, c, k in abc]
            ph = nat.Groth16Phase1(gg1, gg1, gg2, a1[:n], a1[:n], a1[:n], a2[:n], a1[:n - 1])
            nnz = [len(c) for _, c, _ in abc]
            t1, t2 = 2 * nnz[0] + 2 * nnz[1] + nnz[2], nnz[1]
            b1 = j1.repeat((t1 + pool - 1) // pool, 1)[:t1].contiguous()
            b2 = j2.repeat((t2 + pool - 1) // pool, 1)[:t2].contiguous()
            k1, k2 = dev(rand_scalars(t1)), dev(rand_scalars(t2))
            o1, o2 = torch.empty_like(b1), torch.empty_like(b2)

            def new():
                eng.groth16_mpc_new(dabc, n, 4, na, ph, gg1, gg2)

            def wnaf():
                ctx.call_dev("bls_g1_wnaf_mul_dev", b1.data_ptr(), k1.data_ptr(), o1.data_ptr(), t1, 0, eng._stream())
                ctx.call_dev("bls_g2_wnaf_mul_dev", b2.data_ptr(), k2.data_ptr(), o2.data_ptr(), t2, 0, eng._stream())
            t_new, t_wnaf = timed([new, wnaf], args.reps)
            row = {"log_c": log_c, "coefficients": kind, "g1_terms": t1, "g2_terms": t2, "mpc_new_ms": round(t_new, 3),
                   "wnaf_batch_ms": round(t_wnaf, 3), "ratio": round(t_new / t_wnaf, 3),
                   "split_ms": split(new, {"k_mpc_qap": ["k_mpc_qap"], "k_mpc_fix": ["k_mpc_fix"], "normalisation": ["norm", "batch"],
                                           "combine_scan_emit": ["k_mpc_combine", "k_gs_scan", "k_gs_emit", "k_mpc_load"]})}
            res["mpc_new"].append(row)
            print(json.dumps(row), flush=True)
            del b1, b2, k1, k2, o1, o2
    # contribute: h_len + l_len = 2^21
    h_len, l_len = pool - 1, pool
    h = a1[:h_len].contiguous()
    l = a1[:l_len].contiguous()
    params = nat.Groth16Parameters(a1[0], a1[1], a1[2], a2[0], a2[1], h, l, a1[:8], a1[:8], a2[:8], gamma_g2=a2[2], ic=a1[:4],
                                   densities=None, ok=True)
    delta = np.array(rand_scalars(1)[0], dtype=np.uint64)
    bases = torch.cat([j1[:h_len], j1[:l_len]]).contiguous()
    kk = dev(np.repeat(rand_scalars(1), h_len + l_len, 0))
    out = torch.empty_like(bases)

    def contribute():
        eng.groth16_mpc_contribute(params, delta, a1[3].cpu().numpy().view(np.uint64), a2[3].cpu().numpy().view(np.uint64))

    def replicated():
        ctx.call_dev("bls_g1_wnaf_mul_dev", bases.data_ptr(), kk.data_ptr(), out.data_ptr(), h_len + l_len, 0, eng._stream())
    t_c, t_w = timed([contribute, replicated], args.reps)
    res["contribute"] = {"rows": h_len + l_len, "contribute_ms": round(t_c, 3), "replicated_wnaf_ms": round(t_w, 3), "ratio": round(t_c / t_w, 3),
                         "split_ms": split(contribute, {"wnaf": ["wnaf"], "prep": ["k_mpc_prep"], "normalisation": ["norm", "batch"], "emit": ["k_mpc_emit"]})}
    print(json.dumps(res["contribute"]), flush=True)
    # verify: k = 8 contributions on the same key
    after, pks = params, []
    for j in range(8):
        after, pk = eng.groth16_mpc_contribute(after, np.array(rand_scalars(1)[0], dtype=np.uint64), a1[4 + j].cpu().numpy().view(np.uint64),
                                               a2[4 + j].cpu().numpy().view(np.uint64))
        pks.append(pk)
    pks = torch.stack(pks)
    rh, rl = dev(rand_scalars(h_len)), dev(rand_scalars(l_len))
    ok = eng.groth16_mpc_verify(params, after, pks, rh, rl)

    def verify():
        eng.groth16_mpc_verify(params, after, pks, rh, rl)
    (t_v,) = timed([verify], args.reps)
    res["verify"] = {"rows_per_query": pool, "k": 8, "ok": ok, "verify_ms": round(t_v, 3),
                     "split_ms": split(verify, {"multiexp": ["msm", "bucket", "radix", "sort", "Radix"], "pairings": ["miller", "final", "pair", "fq12"],
                                                "compare": ["k_mpcv_diff"]})}
    print(json.dumps(res["verify"]), flush=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    lines = ["Measured with `tools/bench_groth16_mpc.py` on %s (`nvidia-smi` power.limit, clocks.max.sm: %s).  Median of %d calls after a "
             "warm-up, 256 MiB written between calls.\n" % (gpu["name"], gpu["nvidia_smi"], args.reps),
             "| mpc_new | G1 / G2 terms | time | wNAF batch of as many random multiplications | ratio | split (ms) |", "|---|---|---|---|---|---|"]
    for r in res["mpc_new"]:
        lines.append("| 2^%d, %s coefficients | %d / %d | %.1f ms | %.1f ms | %.2f× | %s |" % (r["log_c"], r["coefficients"], r["g1_terms"], r["g2_terms"],
                                                                                 r["mpc_new_ms"], r["wnaf_batch_ms"], r["ratio"], r["split_ms"]))
    c = res["contribute"]
    lines += ["", "| contribute | time | replicated-scalar wNAF | ratio | split (ms) |", "|---|---|---|---|---|",
              "| %d rows | %.1f ms | %.1f ms | %.2f× | %s |" % (c["rows"], c["contribute_ms"], c["replicated_wnaf_ms"], c["ratio"], c["split_ms"])]
    v = res["verify"]
    lines += ["", "| verify | time | ok | split (ms) |", "|---|---|---|---|",
              "| 2^20 rows per query, k = 8 | %.1f ms | %s | %s |" % (v["verify_ms"], v["ok"], v["split_ms"])]
    with open(args.md, "w") as f:
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
