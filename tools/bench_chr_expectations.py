"""ChromosomeNumberMng::computeExpectations on the device: bppgpu_expected_events at the chromosome workload's size (500-taxon
rooted tree, S = 200 counts, one character, one well-conditioned parameter point; tree and data built as bench.py builds the
chromosome_500x4096pts workload), with 10^4 paths per start state (the reference's default) and 10^6.  Reports the device time
of the simulation (with the prefix pass over the tallies) and of the combination with the joint posteriors, the wall time of
the call, paths per second, and the number of simulated events (the class counts of every path at the longest branch).

Baseline: the oracle's vectorised sampler (oracle/ref_mapping.simulate, numpy, one host thread) over a sample of start states,
extrapolated to all 200 of them; labelled as such.  Bio++'s own class is not measured (the reference does not build).

    python tools/bench_chr_expectations.py --out profiles/r8_chr_expectations.json

Needs a B200 (no fallback)."""
from __future__ import annotations

import argparse
import json
import pathlib
import sys
import time

sys.dont_write_bytecode = True
ROOT = pathlib.Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))

import numpy as np  # noqa: E402

from bench_parsimony import card_info  # noqa: E402

SEED = 20260105


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--paths", default="10000,1000000", help="paths per start state, comma separated")
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--baseline-starts", type=int, default=4, help="start states the host baseline simulates")
    ap.add_argument("--baseline-paths", type=int, default=10000)
    a = ap.parse_args()
    from bpp_phyl_b200 import capi, synth
    from oracle import ref_mapping as mp
    import torch
    S, taxa = 200, 500
    rng = np.random.default_rng(SEED)
    tree = synth.random_tree(taxa, rng, mean_brlen=0.02, rooted=True)
    es = synth.chromosome_points(S, 1, seed=SEED + 1000, well_conditioned_only=True)[0]
    gain, loss, dupl, demi = es["params"]
    R = mp.chromosome_classes(1, S, gain=gain, loss=loss, dupl=dupl, demi=demi)
    off = lambda Q: Q * (1 - np.eye(S))
    assert np.array_equal(off(mp.class_sum(R)), off(es["Q"])), "the class split does not add up to the workload's generator"
    md = synth.chromosome_model_desc(es)
    P0, _, _ = capi.pt_batch(md, tree.brlen, capi.WANT_P)
    codes = synth.simulate_single_character(tree, P0, root_state=23, seed=SEED)
    n_unique = int(len(np.unique(codes)))
    tree.brlen = tree.brlen * (n_unique / tree.brlen.sum())      # ChromosomeNumberMng::rescale_tree, as bench.py
    tree.brlen[tree.root] = 0.0
    e = capi.Engine(S, 1, 1, tree.child_off, tree.children, tree.root, np.eye(S),
                    flags=capi.FLAG_KEEP_CLVS | capi.FLAG_WEIGHTED_ROOT)
    e.set_all_tip_codes(codes)
    e.set_pattern_weights(np.ones(1, np.uint32))
    e.set_rates(np.ones(1), np.ones(1))
    e.set_model(0, md)
    e.set_branch_lengths(0, tree.brlen)
    e.set_root_freqs(0, es["pi"])
    lnl, _, _ = e.eval(capi.EVAL_LNL | capi.EVAL_D1)
    lengths = np.array([tree.brlen[n] for n in range(tree.nn) if n != tree.root])
    res = {"card": card_info(), "workload": {"taxa": taxa, "branches": len(lengths), "distinct_lengths": int(len(np.unique(lengths))),
                                             "S": S, "sites": 1, "params": dict(gain=gain, loss=loss, dupl=dupl, demi=demi),
                                             "lnL": float(lnl[0]), "longest_branch": float(lengths.max()),
                                             "tree_length": float(lengths.sum())},
           "device": []}
    e.expected_events(R, 1000, 1)                                 # warm-up: module load, first allocations
    for n in [int(x) for x in a.paths.split(",")]:
        runs = []
        for k in range(a.repeats):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            ex, un = e.expected_events(R, n, SEED + k)
            wall = time.perf_counter() - t0
            sim_ms, comb_ms = capi.expected_events_timing()
            runs.append(dict(wall_s=wall, sim_ms=sim_ms, combine_ms=comb_ms, paths_per_s=S * n / (sim_ms * 1e-3),
                             totals=ex.sum(axis=0).tolist(), unreached_max=float(un.max()), unreached_sum=float(un.sum())))
        _, sums = capi.simulate_event_counts(R, [lengths.max()], n, SEED)
        entry = dict(paths_per_state=n, paths=S * n, events=int(sums.sum()), events_per_path=float(sums.sum()) / (S * n),
                     tally_bytes=int(len(np.unique(lengths)) * S * S * 6 * 8), runs=runs)
        res["device"].append(entry)
        print(json.dumps({k: v for k, v in entry.items() if k != "runs"}), json.dumps(runs[-1]), flush=True)
    starts = np.linspace(0, S - 1, a.baseline_starts).astype(int)
    t0 = time.perf_counter()
    mp.simulate(R, lengths, a.baseline_paths, SEED, starts=starts)
    host = time.perf_counter() - t0
    res["host_baseline"] = {"what": "oracle/ref_mapping.simulate (numpy, one host thread), %d start states x %d paths over all %d lengths; "
                                    "time for 200 states EXTRAPOLATED linearly" % (len(starts), a.baseline_paths, len(lengths)),
                            "measured_s": host, "start_states": starts.tolist(), "paths_per_state": a.baseline_paths,
                            "extrapolated_200_states_s": host * S / len(starts),
                            "paths_per_s": len(starts) * a.baseline_paths / host}
    print(json.dumps(res["host_baseline"]), flush=True)
    pathlib.Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    pathlib.Path(a.out).write_text(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
