"""The parsimony bootstrap at two sizes, DNA simulated under GTR+Gamma4, each search starting from the BIONJ tree:
200 taxa x 20 000 sites with R = 1 000 replicates (a typical bootstrap) and 1024 taxa x 1M sites with R = 16 (the flagship
alignment).  For each size: the sampler's device time, the wall and device time of the lockstep search through the shim
(tools/bench_parsimony_bootstrap.cpp), its rounds and batched calls, and the same replicates searched one after another,
each alone, by the same driver on the same handle and compressed patterns (all of them at the small size, --sequential of
them at the large one); the driver fails unless every such replicate's scores equal the lockstep's.

    python tools/bench_parsimony_bootstrap.py --out profiles/r7_parsimony_bootstrap.json

Needs a B200 (no fallback).  Writes the --out file; the alignment files and the driver go to a temporary directory."""
from __future__ import annotations

import argparse
import json
import pathlib
import subprocess
import sys
import tempfile
import time

sys.dont_write_bytecode = True
ROOT = pathlib.Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))

import numpy as np  # noqa: E402

from bench_parsimony import card_info  # noqa: E402


def build_driver(tmp):
    exe = tmp / "bench_parsimony_bootstrap"
    lib = ROOT / "bpp_phyl_b200" / "lib"
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-I", str(ROOT), "-o", str(exe), str(ROOT / "tools" / "bench_parsimony_bootstrap.cpp"),
                           "-L", str(lib), "-lbppgpu", "-Wl,-rpath," + str(lib)])
    return exe


def run(label, taxa, n_sites, R, n_seq, seed, exe, tmp, res):
    from bpp_phyl_b200 import synth
    from oracle import ref_models as rm
    out = {"taxa": taxa, "sites": n_sites, "replicates": R}
    rng = np.random.default_rng(seed)
    tree = synth.random_tree(taxa, rng, mean_brlen=0.05)
    m = rm.gtr(1.2, 0.8, 0.6, 1.5, 0.9, (.3, .2, .25, .25))
    r, _ = rm.gamma_rates(4, 0.5)
    es = {"Q": m.Q, "V": m.V, "Vinv": m.Vinv, "ev": m.ev_re, "pi": m.freq, "rate": m.rate}
    codes = np.asarray(synth.simulate_tip_codes(tree, es, r, n_sites, seed=seed))       # [L][n_sites], row k = leaf t<k>
    aln = tmp / ("%s.txt" % label)
    lut = np.frombuffer(b"ACGT", np.uint8)
    with open(aln, "wb") as fh:
        for k in range(taxa):
            fh.write(b"t%d " % k)
            fh.write(lut[codes[k]].tobytes())
            fh.write(b"\n")
    t0 = time.perf_counter()
    txt = subprocess.check_output([str(exe), str(aln), str(R), str(seed), str(n_seq)], text=True)
    out["driver_wall_s"] = time.perf_counter() - t0
    lines = txt.splitlines()
    lock = json.loads([l for l in lines if l.startswith("RESULT ")][0][7:])
    scores = lock.pop("scores")
    out["single"] = lock.pop("single")
    out["lockstep"] = lock
    out["lockstep"]["final_scores"] = [s[-1] for s in scores]
    out["lockstep"]["rounds_per_replicate"] = [len(s) - 1 for s in scores]
    sg = out["single"]
    out["per_replicate"] = {
        "lockstep_wall_s": lock["search_wall_s"] / R, "lockstep_device_ms": lock["search_device_ms"] / R,
        "single_wall_s": sg["search_wall_s"] / sg["replicates"], "single_device_ms": sg["search_device_ms"] / sg["replicates"]}
    res[label] = out
    print(label, json.dumps(out["per_replicate"]), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sequential", type=int, default=2, help="replicates run one by one at the large size")
    ap.add_argument("--small-only", action="store_true")
    ap.add_argument("--seed", type=int, default=7)
    ap.add_argument("--out", required=True)
    a = ap.parse_args()
    import __graft_entry__ as g
    g.build()
    res = {"card": card_info()}
    with tempfile.TemporaryDirectory() as d:
        tmp = pathlib.Path(d)
        exe = build_driver(tmp)
        run("200x20k_R1000", 200, 20000, 1000, 1000, a.seed, exe, tmp, res)
        if not a.small_only:
            run("1024x1M_R16", 1024, 1 << 20, 16, a.sequential, a.seed, exe, tmp, res)
    res["card_after"] = card_info()
    pathlib.Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps({k: v for k, v in res.items() if k.startswith("card")}))


if __name__ == "__main__":
    main()
