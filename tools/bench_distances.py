"""Pairwise ML distances + BIONJ at the flagship workload's size (1024 taxa x 1M patterns, GTR+Gamma4): device time per phase,
the int8 operation rate of the count kernel, BIONJ host time, the oracle's single-thread per-pair time extrapolated to all pairs,
and correctness at that size (counts of random pairs against numpy, distances of random pairs against the oracle).

    python tools/bench_distances.py --out profiles/r4_distances_1024x1M.json

Needs a B200 (no fallback).  Writes only the --out file and a temporary directory."""
from __future__ import annotations

import argparse
import json
import os
import pathlib
import subprocess
import sys
import tempfile
import time

for _v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):   # the oracle baseline is single-threaded
    os.environ[_v] = "1"
sys.dont_write_bytecode = True
ROOT = pathlib.Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

import numpy as np  # noqa: E402


def card_info():
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--taxa", type=int, default=1024)
    ap.add_argument("--sites", type=int, default=1 << 20)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--check-count-pairs", type=int, default=1000)
    ap.add_argument("--check-dist-pairs", type=int, default=200)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--out", required=True)
    a = ap.parse_args()

    import __graft_entry__ as g
    g.build()
    sys.path.insert(0, str(ROOT / "tests"))
    import cases
    from bpp_phyl_b200 import capi, synth
    from oracle import ref_distance as rd
    from oracle import ref_models as rm

    res = {"card": card_info(), "taxa": a.taxa, "sites": a.sites, "model": "GTR(1.2,0.8,0.6,1.5,0.9; .3,.2,.25,.25)+Gamma4(0.5)"}
    m = rm.gtr(1.2, 0.8, 0.6, 1.5, 0.9, (.3, .2, .25, .25))
    r, p = rm.gamma_rates(4, 0.5)
    es = {"Q": m.Q, "V": m.V, "Vinv": m.Vinv, "ev": m.ev_re, "pi": m.freq, "rate": m.rate}
    rng = np.random.default_rng(a.seed)
    tree = synth.random_tree(a.taxa, rng, mean_brlen=0.05)
    t0 = time.time()
    codes = synth.simulate_tip_codes(tree, es, r, a.sites, seed=a.seed)          # [L][N] uint8, every site its own pattern
    res["simulate_s"] = time.time() - t0
    w = np.ones(a.sites, np.uint32)
    res["codes_memory"] = "pinned host (as simulate_tip_codes returns them)"
    table = np.eye(4)
    desc = cases.to_model_desc(m)
    L, N, K = a.taxa, a.sites, 4

    def call(counts=False):
        t = time.perf_counter()
        out = capi.pairwise_distances(codes, w, table, desc, m.freq, r, p, counts=counts)
        return out, time.perf_counter() - t

    (d0, l0, cnt), _ = call(counts=True)            # warm-up, and the counts for the checks below
    runs = []
    for _ in range(a.reps):
        (d, l), wall = call()
        up, cm, ml = capi.pairwise_distances_timing()
        assert np.array_equal(d, d0) and np.array_equal(l, l0)
        runs.append({"wall_s": wall, "upload_ms": up, "counts_ms": cm, "ml_ms": ml})
    res["runs"] = runs
    npad = -(-N // 128) * 128
    ops = 2 * 0.5 * (L * K) ** 2 * N
    best = min(x["counts_ms"] for x in runs)
    res["int8_ops_counted"] = ops
    res["int8_ops_note"] = "2 * (L*K)^2 / 2 * N' with N' = %d virtual columns (%d padded); the kernel runs tiles on the diagonal in full" % (N, npad)
    res["counts_tops_best"] = ops / (best * 1e-3) / 1e12
    res["pairs"] = L * (L - 1) // 2

    # BIONJ on the host (the shim's class)
    with tempfile.TemporaryDirectory() as td:
        exe = pathlib.Path(td) / "test_distance"
        lib = ROOT / "bpp_phyl_b200" / "lib"
        subprocess.check_call(["g++", "-std=c++17", "-O2", "-I", str(ROOT), "-o", str(exe), str(ROOT / "tests" / "cpp" / "test_distance.cpp"),
                               "-L", str(lib), "-lbppgpu", "-Wl,-rpath," + str(lib)])
        mf = pathlib.Path(td) / "m.txt"
        with open(mf, "w") as fh:
            fh.write("%d\n" % L)
            for i in range(L):
                fh.write("t%d " % i + " ".join("%.17g" % x for x in d0[i]) + "\n")
        out = subprocess.check_output([str(exe), "bionj", str(mf)], text=True)
        res["bionj_host_ms"] = float(out.split("BIONJ_MS ")[1].split()[0])
        res["bionj_threads"] = os.cpu_count()

    # correctness at this size
    pick = lambda n: [tuple(sorted(rng.choice(L, 2, replace=False))) for _ in range(n)]
    pidx = lambda x, y: x * (2 * L - x - 1) // 2 + (y - x - 1)
    bad = 0
    for x, y in pick(a.check_count_pairs):
        ref = np.bincount(codes[x].astype(np.int64) * K + codes[y], minlength=K * K)
        bad += int(not np.array_equal(cnt[pidx(x, y)].ravel().astype(np.int64), ref))
    res["count_pairs_checked"], res["count_pairs_mismatched"] = a.check_count_pairs, bad
    worst_l, worst_t, n_t, t_or = 0.0, 0.0, 0, []
    for k, (x, y) in enumerate(pick(a.check_dist_pairs)):
        t = time.perf_counter()
        tr, lr = rd.pair_distance(codes[x], codes[y], w, table, m, r, p)
        t_or.append(time.perf_counter() - t)
        worst_l = max(worst_l, abs(l0[x, y] - lr) / abs(lr))
        n = rd.pair_counts(codes[x], codes[y], w, K)
        _, d2 = rd.pair_derivatives(n, table, m, r, p, tr)
        if rd.T_MIN * 1.01 < tr < rd.T_MAX / 1.01 and tr * tr * abs(d2) >= 1.0:
            worst_t = max(worst_t, abs(d0[x, y] - tr) / tr)
            n_t += 1
    res["dist_pairs_checked"] = a.check_dist_pairs
    res["max_rel_lnl_diff"], res["max_rel_t_diff"], res["t_checked"] = worst_l, worst_t, n_t
    res["dist_ok"] = bool(worst_l <= 1e-10 and worst_t <= 1e-6)
    res["oracle_pair_s_median"] = float(np.median(t_or))
    res["oracle_all_pairs_extrapolated_s"] = res["oracle_pair_s_median"] * res["pairs"]
    res["gpu_total_s_best"] = min(x["wall_s"] for x in runs)
    res["card_after"] = card_info()
    pathlib.Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
