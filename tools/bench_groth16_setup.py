"""Groth16 parameter generation (bls_groth16_generate_parameters_dev through DeviceEngine.groth16_generate_parameters) on
one GPU.
Shapes: 2^16, 2^20 and 2^22 constraints (the input constraints included) with num_inputs 4 and 64 and num_aux =
num_constraints - num_inputs, drawn like tests/test_gpu_groth16_setup.py::random_circuit (about 3 terms per linear
combination of A and B, ONE in about half of the constraints, one fresh aux variable per constraint in C), vectorised here
because no witness is needed; coefficients are random canonical values.
Each shape is timed by CUDA events as the median of --reps calls after one warm-up, with a 256 MiB write between calls
(as bench.py does).  In the same process, alternating with the generator, the script times the chain of the existing
calls the generator contains: the two inversions, the ifft of n points, both wNAF tables, the fixed-base exponentiations
over the same numbers of G1 and G2 scalars and both normalisations.  A torch.profiler pass per shape splits the
generator's GPU time by kernel group.  --sweep times the table + fixed-base pair of each group for windows 8 .. 16 at
2^16 and 2^20 (the window the library uses is GS_WINDOW_G1 / GS_WINDOW_G2 of kernels_groth16_setup.cu).
    python tools/bench_groth16_setup.py --out groth16_setup.json --sweep
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "oracle")]

SHAPES = ((16, 4), (16, 64), (20, 4), (20, 64), (22, 4), (22, 64))
WINDOW_G1, WINDOW_G2 = 12, 11          # kernels_groth16_setup.cu


def circuit(log_c, ni, seed):
    """abc as numpy CSR triples, num_aux"""
    rng = np.random.default_rng(seed)
    nc = 1 << log_c
    nq, na = nc - ni, nc - ni
    nv = ni + na
    q = np.arange(nq)
    mats = []
    for k in range(2):
        var = rng.integers(0, ni, size=(nq, 3))
        back = rng.random((nq, 3)) >= 0.3                   # 70 % of the terms on earlier aux variables
        aux = ni + (rng.random((nq, 3)) * np.maximum(q, 1)[:, None]).astype(np.int64)
        var = np.where(back & (q[:, None] > 0), aux, var)
        var[:, 0] = np.where(rng.random(nq) < 0.25, 0, var[:, 0])       # ONE
        mats.append((var.reshape(-1), np.repeat(q, 3)))
    mats.append((ni + q, q))                                            # C: the fresh aux of each constraint
    mats[0] = (np.concatenate([mats[0][0], np.arange(ni)]), np.concatenate([mats[0][1], nq + np.arange(ni)]))
    abc = []
    for var, cons in mats:
        order = np.argsort(var, kind="stable")
        offsets = np.zeros(nv + 1, dtype=np.uint64)
        offsets[1:] = np.cumsum(np.bincount(var, minlength=nv))
        coeff = rng.integers(0, 2 ** 63, size=(len(var), 4), dtype=np.int64).astype(np.uint64)
        coeff[:, 3] &= (1 << 60) - 1
        abc.append((offsets, cons[order].astype(np.uint32), coeff))
    return abc, na


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--sweep", action="store_true")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_groth16_setup.py needs a CUDA device")
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
    g1, g2 = o.generators()
    rng = np.random.default_rng(0x5E7)
    sc = [np.array([int(x) for x in rng.integers(1, 2 ** 62, 4)], dtype=np.uint64) for _ in range(5)]
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a).view(np.int64 if a.dtype == np.uint64 else np.int32)).to(eng.device)
    st = lambda: eng._stream()
    g1j = torch.from_numpy(np.ascontiguousarray(o.g1_from_affine(g1)).view(np.int64)).to(eng.device)
    g2j = torch.from_numpy(np.ascontiguousarray(o.g2_from_affine(g2)).view(np.int64)).to(eng.device)

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

    def exps(g2, window, n, k, out, table):
        t = "g2" if g2 else "g1"
        ctx.call_dev("bls_%s_wnaf_table_dev" % t, (g2j if g2 else g1j).data_ptr(), window, table.data_ptr(), st())
        ctx.call_dev("bls_%s_wnaf_fixed_base_dev" % t, table.data_ptr(), window, k.data_ptr(), out.data_ptr(), n, st())

    def scalars(n):
        x = torch.randint(-(1 << 63), (1 << 63) - 1, (n, 4), dtype=torch.int64, device=eng.device)
        x[:, 3] &= (1 << 60) - 1
        return x

    rows, sweep = [], []
    for lg, ni in SHAPES:
        abc, na = circuit(lg, ni, lg * 100 + ni)
        nc, nv = 1 << lg, ni + na
        dabc = [(dev(off), dev(c), dev(k)) for off, c, k in abc]
        N1, N2 = 3 + nv + (nc - 1) + 2 * nv, 3 + nv
        k1, k2 = scalars(N1), scalars(N2)
        p1 = torch.empty((N1, nat.W_G1), dtype=torch.int64, device=eng.device)
        p2 = torch.empty((N2, nat.W_G2), dtype=torch.int64, device=eng.device)
        t1 = torch.empty((1 << 15, nat.W_G1), dtype=torch.int64, device=eng.device)
        t2 = torch.empty((1 << 15, nat.W_G2), dtype=torch.int64, device=eng.device)
        bn = torch.empty(max(ctx.batch_normalization_scratch_bytes(1, N1), ctx.batch_normalization_scratch_bytes(2, N2)), dtype=torch.uint8, device=eng.device)
        lag = scalars(nc)
        fft_scr = torch.empty(ctx.fr_fft_scratch_bytes(lg, 1), dtype=torch.uint8, device=eng.device)
        gd = scalars(2)
        gi = torch.empty_like(gd)

        def generate():
            return eng.groth16_generate_parameters(dabc, nc, ni, na, g1[0], g2[0], *sc)

        def chain():
            ctx.call_dev("bls_fr_op_dev", nat.OPS["inv"], gd.data_ptr(), None, gi.data_ptr(), None, 2, st())
            ctx.call_dev("bls_fr_fft_dev", nat.FFT_KINDS["ifft"], lag.data_ptr(), lag.data_ptr(), lg, 1, fft_scr.data_ptr(), st())
            exps(False, WINDOW_G1, N1, k1, p1, t1)
            exps(True, WINDOW_G2, N2, k2, p2, t2)
            ctx.call_dev("bls_g1_batch_normalization_dev", p1.data_ptr(), N1, bn.data_ptr(), st())
            ctx.call_dev("bls_g2_batch_normalization_dev", p2.data_ptr(), N2, bn.data_ptr(), st())

        params = generate()
        assert params.ok, "the benchmark circuit has an unconstrained variable"
        a_len, b_len = len(params.a), len(params.b_g1)
        ms_gen, ms_chain = timed([generate, chain], args.reps)
        flush.fill_(1)
        torch.cuda.synchronize()
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            generate()
            torch.cuda.synchronize()
        split = {}
        for ev in prof.key_averages():
            k = ev.key
            grp = ("tables" if "k_wnaf_table" in k else "g2_exp" if "k_wnaf_fixed_base" in k and "Fp2" in k else "g1_exp" if "k_wnaf_fixed_base" in k
                   else "normalisation" if "k_batch_normalization" in k else "qap" if "k_gs_qap" in k else "compaction" if "k_gs_emit" in k or "k_gs_scan" in k
                   else "elementwise" if "k_gs_" in k else "ifft_inv" if ("fft" in k or "fr_op" in k or "k_fr" in k) else "other")
            split[grp] = split.get(grp, 0.0) + ev.self_device_time_total / 1e3
        rows.append({"log_constraints": lg, "num_inputs": ni, "num_aux": na, "nnz": [len(c) for _, c, _ in abc], "a_len": a_len, "b_len": b_len,
                     "g1_exps": N1, "g2_exps": N2, "ms_generate": ms_gen, "ms_chain": ms_chain, "ratio": ms_gen / ms_chain,
                     "profile_ms": split})
        print(json.dumps(rows[-1]), flush=True)
        if args.sweep and ni == 4 and lg in (16, 20):
            for w in range(8, 17):
                g1ms, g2ms = timed([lambda: exps(False, w, N1, k1, p1, t1), lambda: exps(True, w, N2, k2, p2, t2)], 3)
                sweep.append({"log_constraints": lg, "window": w, "g1_exps": N1, "ms_g1_table_and_exps": g1ms, "g2_exps": N2,
                              "ms_g2_table_and_exps": g2ms})
                print(json.dumps(sweep[-1]), flush=True)
        del dabc, k1, k2, p1, p2, t1, t2, bn, lag, fft_scr, params
        eng._scratch.clear()
        torch.cuda.empty_cache()
    res = {"gpu": gpu, "reps": args.reps, "flush_bytes": 256 << 20, "windows": [WINDOW_G1, WINDOW_G2],
           "inputs": "circuit(): seeded numpy CSR; chain scalars torch.randint limbs, top limb masked to 60 bits", "rows": rows, "sweep": sweep}
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    with open(os.path.splitext(args.out)[0] + ".md", "w") as f:
        f.write(markdown(res))


def markdown(res):
    """the tables of profiles/groth16_setup.md from the JSON result"""
    groups = ("tables", "g1_exp", "g2_exp", "normalisation", "ifft_inv", "qap", "elementwise", "compaction", "other")
    out = ["# Groth16 parameter generation (`tools/bench_groth16_setup.py`)", "",
           "%s, `nvidia-smi` power.limit, clocks.max.sm: %s.  Median of %d calls after a warm-up, %d MiB written between calls; "
           "windows G1 %d, G2 %d." % (res["gpu"]["name"], res["gpu"]["nvidia_smi"], res["reps"], res["flush_bytes"] >> 20, *res["windows"]), "",
           "| constraints | num_inputs | G1 / G2 exponentiations | a_len / b_len | generate (ms) | chain of existing calls (ms) | ratio |",
           "|---|---|---|---|---|---|---|"]
    for r in res["rows"]:
        out.append("| 2^%d | %d | %d / %d | %d / %d | %.1f | %.1f | %.3f |" % (r["log_constraints"], r["num_inputs"], r["g1_exps"], r["g2_exps"],
                                                                           r["a_len"], r["b_len"], r["ms_generate"], r["ms_chain"], r["ratio"]))
    out += ["", "GPU time by kernel group, one torch.profiler pass per shape (ms; share of the sum):", "",
            "| constraints | num_inputs | " + " | ".join(groups) + " |", "|---|---|" + "---|" * len(groups)]
    for r in res["rows"]:
        tot = sum(r["profile_ms"].values()) or 1.0
        out.append("| 2^%d | %d | " % (r["log_constraints"], r["num_inputs"]) +
                   " | ".join("%.2f (%.1f %%)" % (r["profile_ms"].get(g, 0.0), 100 * r["profile_ms"].get(g, 0.0) / tot) for g in groups) + " |")
    if res["sweep"]:
        out += ["", "Window sweep: one table build plus the fixed-base exponentiations of the whole batch (ms, median of 3):", "",
                "| constraints | window | G1 (%s) | G2 |" % "scalars as in the rows above", "|---|---|---|---|"]
        for w in res["sweep"]:
            out.append("| 2^%d | %d | %.1f | %.1f |" % (w["log_constraints"], w["window"], w["ms_g1_table_and_exps"], w["ms_g2_table_and_exps"]))
    return "\n".join(out) + "\n"


if __name__ == "__main__":
    main()
