#!/usr/bin/env python
"""bench.py -- the hot path on the BASELINE.json workload, one JSON line on stdout (rank 0).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl native|reference] [--workload NAME] [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A *step* is one full log-likelihood evaluation of the workload (K1 P(t) tables for every branch x class,
K2b tip tables, K2+K3 pruning + root reduction [+ K4/K5 derivatives], and for N > 1 the NCCL all-reduce of the
per-shard scalars).  ``value`` = CLV updates per second (one update = one (node, pattern, class, state) element of
an internal node's conditional likelihood vector, SURVEY.md 8d), whole job, inputs resident in HBM.
``e2e`` = the same through the C-ABI call sequence of one optimiser step with HOST buffers: branch lengths and the
model eigensystem go host->device, log L (and derivatives) come back device->host, inside the timed region.
``--dump-outputs DIR`` writes what the last timed step returned (lnl, and d1 / d2 where the workload asks for them) as
DIR/<name>.npy in float64; the inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark leaves the source tree as it found it
# stdout carries exactly one JSON line: keep NCCL's banner ("NCCL version ...") and any debug output on stderr
os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")

WORKLOADS = {
    # BASELINE.json configs[1]: GTR+G4 DNA, 1024 taxa x 1M patterns
    "dna_gtr_g4_1024x1M": dict(S=4, C=4, taxa=1024, patterns=1_000_000, alpha=0.5, derivs=False, seed=20260102),
    # configs[2]: 20 states + G4, 500 taxa x 200k patterns with d1/d2
    "protein_g4_500x200k_d2": dict(S=20, C=4, taxa=500, patterns=200_000, alpha=0.7, derivs=True, seed=20260103),
    # configs[2] without the derivatives (value-only protein evaluation)
    "protein_g4_500x200k": dict(S=20, C=4, taxa=500, patterns=200_000, alpha=0.7, derivs=False, seed=20260103),
    # layout experiment: the same CLV bytes as protein_g4_500x200k with one class (rows contiguous)
    "protein_c1_500x800k": dict(S=20, C=1, taxa=500, patterns=800_000, alpha=None, derivs=False, seed=20260103),
    # configs[3]: 64-state codon (61 sense + 3 inert stop lines), 200 taxa x 100k patterns, C = 1: YN98 and GY94
    "codon_200x100k": dict(S=64, C=1, taxa=200, patterns=100_000, alpha=None, derivs=False, seed=20260104, model="YN98"),
    "codon_gy94_200x100k": dict(S=64, C=1, taxa=200, patterns=100_000, alpha=None, derivs=False, seed=20260104, model="GY94"),
    # configs[4]: ChromEvol-style chromosome-number model, 200 states, 500 taxa, one character, 4096 parameter points
    "chromosome_500x4096pts": dict(S=200, C=1, taxa=500, patterns=1, points=4096, alpha=None, derivs=False, seed=20260105),
}
DEFAULT = "dna_gtr_g4_1024x1M"


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# stdout must carry exactly ONE JSON line.  Native libraries write banners to file descriptor 1 whatever Python does (NCCL's
# "NCCL version ..." from the communicator the engine creates): keep a private copy of the real stdout for the JSON line and
# point descriptor 1 at stderr for everything else.
_JSON_OUT = None


def _claim_stdout():
    global _JSON_OUT
    if _JSON_OUT is None:
        sys.stdout.flush()
        _JSON_OUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line):
    _claim_stdout()
    _JSON_OUT.write(json.dumps(line) + "\n")
    _JSON_OUT.flush()


DUMP_BYTES = 64 << 20


def dump_outputs(d, arrays):
    """d/<name>.npy (float64) for every array, DUMP_BYTES in all: an array over its share is replaced by the same seeded sample
    of its flattened entries on every run."""
    os.makedirs(d, exist_ok=True)
    share = DUMP_BYTES // 8 // len(arrays)
    for name, x in arrays.items():
        x = np.asarray(x, np.float64)
        if x.size > share:
            x = x.ravel()[np.sort(np.random.default_rng(0).choice(x.size, share, replace=False))]
        np.save(os.path.join(d, name + ".npy"), x)
    log("outputs of the last timed step written to %s: %s" % (d, ", ".join(sorted(arrays))))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, pw = [], [], set(), []
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2])); pw.append(float(r[3]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


def algorithmic_bytes(tree, N, C, S):
    """SURVEY.md 8d: per CLV update at a node with k sons of which k_t are tips: 8*(1 + k - k_t) bytes."""
    tot = 0
    for n in range(tree.nn):
        sons = tree.sons(n)
        if len(sons) == 0:
            continue
        k_int = int((~tree.is_leaf[sons]).sum())
        tot += 8 * (1 + k_int)
    return tot * N * C * S


def model_for(w, rng):
    """The workload's substitution model, built by the product's own C++ host code (bppgpu_host_model: generator +
    updateMatrices): GTR for DNA, LG08 for protein, YN98 / GY94 (64 states, three inert stop lines) for codons."""
    from bpp_phyl_b200 import capi
    if w["S"] == 4:
        return capi.host_model("GTR", 1.2, 0.8, 0.6, 1.5, 0.9, .3, .2, .25, .25)
    if w["S"] == 20:
        return capi.host_model("LG08")
    if w.get("model") == "GY94":
        return capi.host_model("GY94", 2.0, 80.0)
    return capi.host_model("YN98", 2.0, 0.3)


def build_inputs(w, rank, world, device):
    """Tree + model + this rank's contiguous pattern shard (strong scaling: the workload's patterns are split)."""
    from bpp_phyl_b200 import synth
    rng = np.random.default_rng(w["seed"])
    tree = synth.random_tree(w["taxa"], rng, mean_brlen=0.05)
    es = model_for(w, rng)
    rates, probs = synth.gamma_rates(w["C"], w["alpha"]) if w["C"] > 1 else (np.ones(1), np.ones(1))
    N = w["patterns"]
    from bpp_phyl_b200.shard import shard_range
    lo, hi = shard_range(N, rank, world)
    t0 = time.time()
    nblk = 16
    if N % nblk == 0 and nblk % world == 0 and N >= nblk:
        # world-size invariant data: the job's patterns are 16 independently seeded blocks and a rank simulates the blocks
        # of its range, so strong-scaling runs at 1, 2, 4, 8 GPUs evaluate the SAME alignment (equal lnL is then a full-size
        # check of the sharding)
        B = N // nblk
        b0 = lo // B
        parts = [synth.simulate_tip_codes(tree, es, rates, B, seed=w["seed"] + 7919 * (b0 + k + 1), device=device)
                 for k in range((hi - lo) // B)]
        codes = np.concatenate(parts, axis=1) if len(parts) > 1 else parts[0]
    else:
        codes = synth.simulate_tip_codes(tree, es, rates, hi - lo, seed=w["seed"] + 7919 * rank, device=device)
    log("[rank %d] simulated %d patterns x %d tips in %.1fs" % (rank, hi - lo, tree.n_leaves, time.time() - t0))
    return tree, es, rates, probs, codes


def make_engine(w, tree, es, rates, probs, codes, dev_index, flags):
    from bpp_phyl_b200 import capi, synth
    S = w["S"]
    e = capi.Engine(S, w["C"], codes.shape[1], tree.child_off, tree.children, tree.root, np.eye(S), device=dev_index,
                    flags=flags)
    e.set_all_tip_codes(codes)
    e.set_pattern_weights(np.ones(codes.shape[1], np.uint32))
    e.set_rates(rates, probs)
    md = synth.model_desc(es)
    e.set_model(0, md)
    e.set_branch_lengths(0, tree.brlen)
    e.set_root_freqs(0, es["pi"])
    return e, md


def _cpu_args(w, tree, es, rates, probs, sub, want, threads):
    n = sub.shape[1]
    return dict(S=w["S"], Ccat=w["C"], N=n, child_off=tree.child_off, children=tree.children, root=tree.root, codes=sub,
                code_table=np.eye(w["S"]), weights=np.ones(n, np.uint32), rates=rates, probs=probs, V=es["V"],
                Vinv=es["Vinv"], ev=es["ev"], model_rate=es.get("rate", 1.0), brlen=tree.brlen, rootfreq=es["pi"], scaled=True,
                want=want, nthreads=threads)


def cpu_leg(w, tree, es, rates, probs, codes, lnl_gpu_full, budget_s=60.0):
    """The reference's CPU algorithm (oracle/ref_cpu.cpp, a port: the reference cannot be built here) on the SAME simulated
    data as the GPU run, three ways (SURVEY 8d): one thread (what the reference is), 8 threads and all host threads as
    independent pattern shards -- each on a bounded sample -- and, inside the time budget, the FULL input in blocks for the
    full-size parity check (lnL summed over the blocks against the GPU's lnL of the whole input)."""
    from oracle import ref_cpu
    ref_cpu.build()
    cores = os.cpu_count() or 1
    N = codes.shape[1]
    want = 7 if w["derivs"] else 1
    per_upd = tree.n_internal * w["C"] * w["S"]
    out = {"unit": "CLV updates/s", "kind": "port", "cores": cores}

    def run(n, threads, wnt):
        sub = np.ascontiguousarray(codes[:, :n])
        r = ref_cpu.eval_raw(reps=1, **_cpu_args(w, tree, es, rates, probs, sub, wnt, threads))
        return r, sub

    per_thread = 256 if w["S"] >= 20 else 512
    r1, _ = run(min(N, per_thread), 1, want)
    out["one_thread"] = {"value": per_upd * min(N, per_thread) / r1["seconds"], "cores": 1,
                         "sample": "%d patterns, full tree, %.2f s" % (min(N, per_thread), r1["seconds"])}
    if cores >= 8:
        n8 = min(N, per_thread * 8)
        r8, _ = run(n8, 8, want)
        out["eight_shards"] = {"value": per_upd * n8 / r8["seconds"], "cores": 8,
                               "sample": "%d patterns as 8 independent pattern shards, %.2f s" % (n8, r8["seconds"])}
    nall = min(N, per_thread * cores)
    rall, sub = run(nall, cores, want)
    out["value"] = per_upd * nall / rall["seconds"]
    out["sample"] = "%d of %d patterns (the GPU run's own data), full tree, %d host threads as independent pattern shards, " \
                    "%.2f s, scaled arithmetic%s" % (nall, N, cores, rall["seconds"], ", with d1/d2" if w["derivs"] else "")
    out["lnl_sample"] = rall["lnl"]
    # full-size parity, value only: whole input in blocks of `blk` patterns, if the extrapolated time fits the budget
    t_full = rall["seconds"] * N / nall * (0.45 if w["derivs"] else 1.0)
    parity = {"lnl_gpu_full": lnl_gpu_full, "patterns": N}
    if t_full <= budget_s or os.environ.get("BPPGPU_BENCH_FULL_PARITY") == "1":
        blk = per_thread * cores
        t0 = time.time()
        tot, secs = ref_cpu.eval_blocks(w["S"], w["C"], N, blk, tree.child_off, tree.children, tree.root, codes, np.eye(w["S"]),
                                        np.ones(N, np.uint32), rates, probs, es["V"], es["Vinv"], es["ev"], es.get("rate", 1.0),
                                        tree.brlen, es["pi"], scaled=True, nthreads=cores)
        log("full-size CPU parity: %.1f s evaluation, %.1f s wall" % (secs, time.time() - t0))
        parity.update({"lnl_cpu_full": tot, "rel_diff_full": abs(tot - lnl_gpu_full) / abs(tot), "cpu_seconds_full": secs,
                       "cpu_updates_per_s_full": per_upd * N / secs,
                       "note": "CPU port over the whole input in blocks of %d patterns on %d threads (arrays allocated once); lnL summed over blocks" % (blk, cores)})
    else:
        parity.update({"lnl_cpu_full": None, "rel_diff_full": None,
                       "note": "full input would take %.0f s on %d threads (> %.0f s budget): sample parity only; "
                               "set BPPGPU_BENCH_FULL_PARITY=1 to force" % (t_full, cores, budget_s)})
    return out, sub, parity


def ncu_traffic(kernel):
    """dram__bytes_read.sum + dram__bytes_write.sum of one launch of `kernel`, from the committed ncu summaries (profiles/);
    None when no capture of that kernel on this workload is committed."""
    import csv
    import glob
    best = None
    for f in sorted(glob.glob(os.path.join(ROOT, "profiles", "*_ncu_summary.csv"))):
        rd = wr = None
        try:
            for row in csv.reader(open(f)):
                if len(row) == 4 and kernel.split("_kernel")[0] in row[0]:
                    scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}.get(row[2])
                    if row[1] == "dram__bytes_read.sum" and scale and rd is None:
                        rd = float(row[3]) * scale
                    if row[1] == "dram__bytes_write.sum" and scale and wr is None:
                        wr = float(row[3]) * scale
        except OSError:
            continue
        if rd is not None and wr is not None and kernel in ("walk4_kernel", "walk4c_kernel"):
            best = rd + wr          # the walk captures are of the default (1M-pattern) workload; the latest file wins
    return best


def ncu_traffic_per_eval(workload, kernel):
    """DRAM bytes of all launches of `kernel` in one evaluation of `workload` (profiles/r1e_traffic.json, written by
    tools/traffic_from_launches.py from the committed ncu launch list), or None."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "r1e_traffic.json")))
        return t[workload][kernel]["dram_bytes_per_eval"]
    except (OSError, ValueError, KeyError):
        return None


def family_dmma_flops(tree, rows):
    """FP64 tensor-core flops the per-father derivative kernel issues (S = 20, d1 + d2): per 8 rows and class, 15 DMMAs
    (m8n8k4, 512 flop) for the father contraction of every non-root father and 40 per internal son (P | dP | d2P stacked)."""
    dmma = 0
    for n in range(tree.nn):
        sons = tree.sons(n)
        if not len(sons):
            continue
        dmma += (15 if n != tree.root else 0) + 40 * sum(1 for s in sons if len(tree.sons(s)))
    return dmma * 512.0 * rows / 8


def flops_per_eval(tree, rows, S):
    """pruning contraction flops: 2 S^2 per (row, internal son) + S per extra son (SURVEY 8d)"""
    tot = 0
    for n in range(tree.nn):
        sons = tree.sons(n)
        if len(sons) == 0:
            continue
        k_int = int((~tree.is_leaf[sons]).sum())
        tot += k_int * 2 * S * S + (len(sons) - 1) * S
    return tot * rows


def run_points(a, w, rank, world, local, K, W, metric, config):
    """configs[4]: many parameter points on one character.  Points are an independent batch axis: each rank takes a
    contiguous block of them, no collective (DESIGN.md section 6)."""
    import torch
    import torch.distributed as dist
    from bpp_phyl_b200 import capi, synth
    from bpp_phyl_b200.shard import shard_range
    device = "cuda:%d" % local
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(device))
    S = w["S"]
    npts_total = (a.points or w["points"]) * (world if a.scaling == "weak" else 1)
    lo, hi = shard_range(npts_total, rank, world)
    npts = hi - lo
    rng = np.random.default_rng(w["seed"])
    tree = synth.random_tree(w["taxa"], rng, mean_brlen=0.02, rooted=True)
    t0 = time.time()
    # every point drawn from the box stays in the batch, on the route the reference takes for it (synth.chromosome_eigensystem):
    # eigen form where V can be inverted, Taylor series + squaring otherwise; --well-conditioned restores the round-1 sample
    pts = synth.chromosome_points(S, npts, seed=w["seed"] + 1000 * rank, well_conditioned_only=a.well_conditioned)
    n_series = sum(1 for es in pts if es["route"] == "series")
    n_illcond = sum(1 for es in pts if es["route"] == "eigen" and es["resid"] > 1e-9)
    good = [k for k, es in enumerate(pts) if es["route"] == "eigen" and es["resid"] <= 1e-9]
    if not good:   # (a handful of points and none well-conditioned: simulate and sample on whatever has an eigen form)
        good = [k for k, es in enumerate(pts) if es["route"] == "eigen"] or [0]
    log("[rank %d] %d parameter points (host eigendecompositions) in %.1fs: %d series route, %d eigen route with |V D V^-1 - Q| > 1e-9 |Q|, %d well-conditioned"
        % (rank, npts, time.time() - t0, n_series, n_illcond, len(good)))
    mds = [synth.chromosome_model_desc(es) for es in pts]
    P0, _, _ = capi.pt_batch(mds[good[0]], tree.brlen, capi.WANT_P, device=local)   # the data are simulated under a well-conditioned point
    codes = synth.simulate_single_character(tree, P0, root_state=23, seed=w["seed"])
    # ChromosomeNumberMng::rescale_tree (App/ChromosomeNumberMng.cpp:121-147, branchMul_ = 999): the total tree length becomes the
    # number of distinct chromosome counts in the data before anything is evaluated
    n_unique = int(len(np.unique(codes)))
    tree.brlen = tree.brlen * (n_unique / tree.brlen.sum())
    tree.brlen[tree.root] = 0.0
    e = capi.Engine(S, 1, 1, tree.child_off, tree.children, tree.root, np.eye(S), n_points=npts, n_models=npts, device=local,
                    flags=capi.FLAG_WEIGHTED_ROOT)
    e.set_all_tip_codes(codes)
    e.set_pattern_weights(np.ones(1, np.uint32))
    e.set_rates(np.ones(1), np.ones(1))
    for k in range(npts):
        e.set_model(k, mds[k])
        e.set_branch_lengths(k, tree.brlen)
    nn = tree.nn
    out = torch.zeros(npts * (1 + 2 * nn), dtype=torch.float64, device=device)
    stream = torch.cuda.Stream(device=device)
    torch.cuda.set_stream(stream)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    log("[rank %d] engine ready, path %d" % (rank, e.stats()["path"]))
    for _ in range(W):
        e.eval_device(1, out.data_ptr(), stream.cuda_stream)
    barrier()
    e.stats()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record(stream)
    for _ in range(K):
        e.eval_device(1, out.data_ptr(), stream.cuda_stream)
    ev1.record(stream)
    barrier()
    if a.dump_outputs:
        lnl_pts = out.view(npts, 1 + 2 * nn)[:, 0].cpu().numpy()
        if world > 1:
            parts = [None] * world
            dist.all_gather_object(parts, lnl_pts)
            lnl_pts = np.concatenate(parts)
        if rank == 0:
            dump_outputs(a.dump_outputs, {"lnl": lnl_pts})
    ms = ev0.elapsed_time(ev1)
    st = e.stats()
    log("[rank %d] timed region done: %.3f ms/step, P(t) %.3f ms, pruning %.3f ms" % (rank, ms / K, st["pt_ms_sum"] / K, st["prune_ms_sum"] / max(1, st["prune_count"])))
    lnl0 = float(out[good[0] * (1 + 2 * nn)].item())
    # e2e: every point's model (host eigensystem) and branch lengths go host -> device, log L of every point comes back
    # per point: the head of the model image [V | V^-1 | re | im | role] (the generator is not read by any route of these models
    # and does not travel) + the branch lengths
    head = ((2 * S * S + 2 * S + (S + 1) // 2 + 31) // 32 * 32) * 8
    h2d = (npts - n_series) * head + n_series * (head + 2 * S * S * 8) + npts * nn * 8   # (series models travel with Q and Q^2)
    d2h = npts * 8

    def step_e2e():
        e.set_models(0, mds)                       # every point's eigensystem, host -> device (pinned staging)
        for k in range(npts):
            e.set_branch_lengths(k, tree.brlen)
        return e.eval(1)[0]

    n_e2e = 0 if a.profile else max(1, min(K, 2))
    barrier()
    t0 = time.perf_counter()
    for _ in range(n_e2e):
        lnl_host = step_e2e()
    barrier()
    e2e_ms = 1e3 * (time.perf_counter() - t0) / max(1, n_e2e)
    tms = torch.tensor([ms, e2e_ms], dtype=torch.float64, device=device)
    if world > 1:
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
    ms, e2e_ms = float(tms[0]), float(tms[1])
    dfma_now, dmma_now = capi.measure_fp64_peak(local) if rank == 0 else (None, None)
    clocks = sampler.stop() if rank == 0 else None
    upd_step = tree.n_internal * npts_total * S          # CLV updates of the whole job per step
    if rank == 0:
        dmma_peak = dmma_now
        kms = st["prune_ms_sum"] / max(1, st["prune_count"])      # level kernels + root (factored) or node kernels (tables)
        pt_ms = st["pt_ms_sum"] / max(1, K)                        # guard (factored) or all P(t) chunks (tables)
        nfac, ntab = int(st["factored_points"]), int(st["table_points"])
        if ntab > 0:
            # points on the table route (Taylor series / clamped eigen tables) dominate the batch: the step is the P(t) launches of
            # those points (pt_series_kernel<DMMA>, pt_dmma_kernel); their DMMA count depends on the terms and squarings of every
            # branch and is not tallied, so the fraction comes from ncu (profiles/), not from this line
            roofline = {"bound": "tensor", "kernel": "pt_series_kernel<DMMA> (Taylor + squaring, one CTA per branch matrix) + pt_dmma_kernel of the "
                                                     "guard-failed points",
                        "achieved": None, "peak": dmma_peak, "unit": "TFLOP/s", "frac": None, "traffic": None,
                        "kernel_ms": pt_ms, "peak_source": "FP64 mma.sync m8n8k4 measured in this run (bppgpu_measure_fp64_peak)",
                        "note": "kernel_ms = all P(t) launches of the step (guard probes + tables of the table-route points), event timed; "
                                "DMMA pipe of pt_series_kernel<DMMA> in ncu: profiles/r2b_pt_series_dmma_2cta_metrics.csv"}
        elif nfac > 0:
            K8 = (S + 7) // 8 * 8
            dm_flops = nfac * (st["chr_cblocks_tip"] + 2 * st["chr_cblocks_dense"]) * (K8 // 8) * (K8 // 4) * 512.0
            ach = dm_flops / (kms * 1e-3) / 1e12 if kms > 0 else None
            roofline = {"bound": "tensor", "kernel": "chr_level_kernel / chr_chain_kernel (one launch per wide tree level, one for the single-tile levels above; all levels + root timed together)",
                        "achieved": ach, "peak": dmma_peak, "unit": "TFLOP/s", "frac": ach / dmma_peak if ach else None, "traffic": None,
                        "kernel_ms": kms, "executed_dmma_flops_per_eval": dm_flops, "guard_ms": pt_ms,
                        "peak_source": "FP64 mma.sync m8n8k4 measured in this run (bppgpu_measure_fp64_peak)",
                        "note": "P(t) is applied in factored form V T(t) V^-1 x, tree level by tree level, as skinny tensor-core GEMMs; "
                                "flops = DMMAs issued x 512 (only the 8-column blocks in use are issued)"}
        else:
            n_mat = npts * (nn - 1)
            flops = n_mat * (2.0 * S ** 3 + S * S)
            ach = flops / (pt_ms * 1e-3) / 1e12 if pt_ms > 0 else None
            roofline = {"bound": "tensor", "kernel": "pt_dmma_kernel", "achieved": ach, "peak": dmma_peak, "unit": "TFLOP/s",
                        "frac": ach / dmma_peak if ach else None, "traffic": None, "kernel_ms": pt_ms, "flops_per_eval": flops,
                        "node_kernels_ms": kms,
                        "peak_source": "FP64 mma.sync m8n8k4 measured in this run (bppgpu_measure_fp64_peak)"}
        line = {"metric": metric, "value": upd_step * K / (ms * 1e-3), "unit": "CLV updates/s", "n_gpus": world, "steps": K,
                "warmup": W, "ms_per_step": ms / K, "higher_is_better": True, "scaling": a.scaling, "vs_baseline": None,
                "dtype": "f64", "data": "synthetic (one chromosome count per taxon simulated down a random rooted tree; parameter points "
                                        "drawn uniformly from gain, loss in (0, 2), dupl, demi in (0, 1); " +
                                        ("numerically defective generators redrawn (--well-conditioned)" if a.well_conditioned else
                                         "every drawn point kept, on the route the reference takes for it") + ")",
                "config": dict(config, points=npts_total, sharding="points/%d (replicas, no collective)" % world,
                               tree_length="rescaled to the %d distinct counts of the data (rescale_tree)" % n_unique),
                "logl_evals_per_s": npts_total * K / (ms * 1e-3), "lnl_point0": lnl0,
                "points_drawn": {"series_route": n_series, "eigen_route_illconditioned": n_illcond, "eigen_route_wellconditioned": len(good),
                                 "rule": "series = V not invertible (non-finite inverse or cond(V) > 1e15) or no unique null eigenvalue, as "
                                         "ChromosomeSubstitutionModel.cpp:686-767 decides; ill-conditioned = eigen route whose V D V^-1 misses Q by "
                                         "more than 1e-9 max|Q| (the reference never checks and still uses it)"},
                "routes": {"factored_points": nfac, "table_points": ntab,
                           "note": "points whose probe tables leave [0, 1] by more than 1e-8 (where the reference's per-entry clamp would matter) "
                                   "and singular generators take the P-table route"},
                "e2e": {"value": upd_step / (e2e_ms * 1e-3) if e2e_ms > 0 else None, "unit": "CLV updates/s",
                        "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms,
                        "logl_evals_per_s": npts_total / (e2e_ms * 1e-3) if e2e_ms > 0 else None,
                        "call": "bppgpu_set_models (all points) + bppgpu_set_branch_lengths per point, one bppgpu_eval (host buffers); the host "
                                "eigendecompositions are NOT inside (see host_eigen)"},
                "gpu_launches": int(st["kernel_launches"]) * K, "launches_per_step": int(st["kernel_launches"]),
                "roofline": roofline, "clocks": clocks, "fp64_peaks_measured": {"dfma_tflops": dfma_now, "dmma_m8n8k4_tflops": dmma_now},
                "hbm_resident_bytes": int(st["hbm_bytes_resident"])}
        # the host side of a model update: ChromosomeSubstitutionModel::updateMatrices / updateEigenMatrices through the C++
        # shim (bppgpu_host_model), one thread, a few points -- the reference pays this (plus 30 matrix powers) per point and step
        t0 = time.perf_counter()
        nh = min(4, npts)
        for es in pts[:nh]:
            g_, l_, du_, de_ = es["params"]
            capi.host_model("Chromosome", 1, S, g_, l_, du_, de_)
        line["host_eigen"] = {"shim_ms_per_model_one_thread": 1e3 * (time.perf_counter() - t0) / nh, "models_timed": nh,
                              "note": "outside every timed region; the bench's eigensystems come from numpy (LAPACK) before the run"}
        if world == 1 and not a.no_cpu:
            # the reference's CPU algorithm on a few points, one point per host thread
            from concurrent.futures import ThreadPoolExecutor
            from oracle import ref_cpu
            ref_cpu.build()
            threads = min(os.cpu_count() or 1, len(good), 16)

            def one(j):
                es = pts[good[j]]
                return ref_cpu.eval_raw(S, 1, 1, tree.child_off, tree.children, tree.root, codes, np.eye(S), np.ones(1, np.uint32),
                                        np.ones(1), np.ones(1), es["V"], es["Vinv"], es["ev"], 1.0, tree.brlen, es["pi"], scaled=True,
                                        want=1, nthreads=1, reps=1, ev_im=es["ev_im"], chr_clamp=True, weighted_root=True)
            t0 = time.perf_counter()
            with ThreadPoolExecutor(threads) as ex:
                res = list(ex.map(one, range(threads)))
            dt = time.perf_counter() - t0
            rel = max(abs(res[j]["lnl"] - lnl_host[good[j]]) / abs(res[j]["lnl"]) for j in range(threads))
            line["cpu_baseline"] = {"value": tree.n_internal * threads * S / dt, "unit": "CLV updates/s", "cores": threads, "kind": "port",
                                    "sample": "the first %d well-conditioned eigen-route points of %d, full tree, one point per thread, %.1f s"
                                              % (threads, npts_total, dt),
                                    "logl_evals_per_s": threads / dt, "rel_diff_vs_gpu": rel}
        emit(line)
        log("[rank 0] JSON line printed")
    e.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None,
                    help="timed steps (default 20; 3 for the chromosome workload on the whole parameter box, whose step takes ~16 s)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--workload", default=DEFAULT, choices=sorted(WORKLOADS))
    ap.add_argument("--patterns", type=int, default=0, help="override the workload's pattern count (debug)")
    ap.add_argument("--points", type=int, default=0, help="override the number of parameter points (chromosome workload)")
    ap.add_argument("--scaling", default="strong", choices=["weak", "strong"],
                    help="N > 1: strong (default, BASELINE's north-star) = the workload's patterns are split across the GPUs; "
                         "weak = every GPU gets the workload's pattern count.  A strong run also times the weak job and reports it "
                         "under the key `weak` of the same line.")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--well-conditioned", action="store_true",
                    help="chromosome workload: redraw parameter points whose eigen form misses the generator (the round-1 sample)")
    ap.add_argument("--no-weak", action="store_true", help="N > 1: skip the weak-scaling job timed after the strong one")
    ap.add_argument("--profile", action="store_true", help="1 warm-up + 1 timed step, no e2e / CPU legs (for ncu only)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned to DIR/<name>.npy (float64, at most 64 MB in all)")
    a = ap.parse_args()
    if a.steps is not None and a.steps < 1:
        ap.error("--steps must be at least 1")
    _claim_stdout()
    w = dict(WORKLOADS[a.workload])
    if a.patterns:
        w["patterns"] = a.patterns
    W = max(a.warmup, 3) if a.impl == "native" else a.warmup
    K = a.steps if a.steps else (3 if ("points" in w and not a.well_conditioned) else 20)
    if a.profile:
        W, K, a.no_cpu = 1, 1, True
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    per_gpu_patterns = w["patterns"]
    if a.scaling == "weak" and "points" not in w:
        w["patterns"] = per_gpu_patterns * world        # whole job; each rank still owns a contiguous 1/world block
    metric = "CLV updates/s"
    config = {"workload": a.workload, "states": w["S"], "rate_classes": w["C"], "taxa": w["taxa"],
              "patterns": w["patterns"], "patterns_per_gpu": w["patterns"] // world, "derivatives": w["derivs"],
              "sharding": "contiguous pattern blocks, one per GPU; NCCL all-reduce of (lnL, d1, d2) inside the engine (bppgpu_comm_init)",
              "l2": "inputs larger than L2 (tip codes %.0f MB per rank; CLVs never re-read from a previous step)" %
                    (w["taxa"] * w["patterns"] / world / 1e6)}

    if "points" in w and a.impl == "native":
        import __graft_entry__ as g
        from bpp_phyl_b200 import capi
        if not capi.LIB_PATH.exists():
            g.build_lib()
        return run_points(a, w, rank, world, local, K, W, metric, config)
    if a.impl == "reference":
        if rank != 0:
            return 0
        from bpp_phyl_b200 import synth
        rng = np.random.default_rng(w["seed"])
        tree = synth.random_tree(w["taxa"], rng, mean_brlen=0.05)
        es = model_for(w, rng)         # host code only (bppgpu_host_model launches nothing)
        rates, probs = synth.gamma_rates(w["C"], w["alpha"]) if w["C"] > 1 else (np.ones(1), np.ones(1))
        threads = os.cpu_count() or 1
        n = (256 if w["S"] >= 20 else 512) * threads
        # the native arm's data-generating process (tips simulated down the tree under the model), sampled on the CPU
        codes = synth.simulate_tip_codes(tree, es, rates, n, seed=w["seed"] + 7919, device="cpu")
        from oracle import ref_cpu
        ref_cpu.build()
        want = 7 if w["derivs"] else 1
        args = _cpu_args(w, tree, es, rates, probs, codes, want, threads)
        # one call: W + K evaluations on the same likelihood object (setData-style allocation is not part of a step);
        # the C side times every evaluation, the last K are the timed steps
        if a.warmup:
            ref_cpu.eval_raw(reps=max(1, a.warmup), **args)
        r = ref_cpu.eval_raw(reps=K, **args)
        if a.dump_outputs:
            dump_outputs(a.dump_outputs, {"lnl": [r["lnl"]], "d1": r["d1"], "d2": r["d2"]} if w["derivs"] else {"lnl": [r["lnl"]]})
        dt = r["total_seconds"]
        upd = tree.n_internal * n * w["C"] * w["S"]
        val = upd * K / dt
        r1 = ref_cpu.eval_raw(reps=1, **_cpu_args(w, tree, es, rates, probs, np.ascontiguousarray(codes[:, :n // threads]), want, 1))
        one = tree.n_internal * (n // threads) * w["C"] * w["S"] / r1["seconds"]
        sample = "%d of %d patterns per step (full tree, tips simulated under the model like the native arm's), %d host threads as " \
                 "independent pattern shards" % (n, w["patterns"], threads)
        emit({"impl": "reference", "metric": metric, "value": val, "unit": "CLV updates/s", "n_gpus": a.gpus,
                          "steps": K, "warmup": a.warmup, "ms_per_step": 1e3 * dt / K, "higher_is_better": True,
                          "scaling": a.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                          "config": config,
                          "cpu_baseline": {"value": val, "unit": "CLV updates/s", "cores": threads, "kind": "port", "sample": sample,
                                           "one_thread": {"value": one, "cores": 1,
                                                          "sample": "%d patterns, %.2f s" % (n // threads, r1["seconds"])}},
                          "e2e": {"value": val, "unit": "CLV updates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})
        return 0

    # ---------------- native arm ----------------
    import torch
    import torch.distributed as dist
    import __graft_entry__ as g
    from bpp_phyl_b200 import capi, shard
    if not capi.LIB_PATH.exists():
        g.build_lib()
    torch.cuda.set_device(local)
    device = "cuda:%d" % local
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(device))
    flags = capi.FLAG_KEEP_CLVS if w["derivs"] else 0
    want = 7 if w["derivs"] else 1
    tree, es, rates, probs, codes = build_inputs(w, rank, world, device)
    e, md = make_engine(w, tree, es, rates, probs, codes, local, flags)
    nn = tree.nn
    out = torch.zeros(1 + 2 * nn, dtype=torch.float64, device=device)
    # a real (non-NULL) stream: kernels, NCCL and the timing events all go on it
    stream = torch.cuda.Stream(device=device)
    torch.cuda.set_stream(stream)

    if world > 1:
        shard.join_engine(e, device)   # bppgpu_comm_init: the engine all-reduces (lnL, d1, d2) itself, on the evaluation's stream

    def step_device():
        e.eval_device(want, out.data_ptr(), stream.cuda_stream)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    log("[rank %d] engine ready, path %d" % (rank, e.stats()["path"]))
    for _ in range(W):
        step_device()
    barrier()
    log("[rank %d] warm-up done" % rank)
    st0 = e.stats()             # clears the kernel-timing ring
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record(stream)
    for _ in range(K):
        step_device()
    ev1.record(stream)
    barrier()
    if a.dump_outputs and rank == 0:
        res = out.cpu().numpy()          # every rank holds the whole alignment's result row
        dump_outputs(a.dump_outputs, {"lnl": res[:1], "d1": res[1:1 + nn], "d2": res[1 + nn:]} if w["derivs"] else {"lnl": res[:1]})
    ms = ev0.elapsed_time(ev1)
    log("[rank %d] timed region done: %.3f ms/step" % (rank, ms / K))
    st = e.stats()
    lnl_dev = float(out[0].item())
    tms = torch.tensor([ms], dtype=torch.float64, device=device)
    if world > 1:
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
    ms = float(tms.item())

    # ---- e2e: one optimiser step through the C ABI with host buffers -----------------------------------------
    brl = tree.brlen.copy()
    host_out = torch.empty(1 + 2 * nn, dtype=torch.float64).pin_memory()
    h2d = brl.nbytes + es["V"].nbytes + es["Vinv"].nbytes + es["ev"].nbytes + es["Q"].nbytes
    d2h = 8 * (1 + (2 * nn if w["derivs"] else 0))

    def step_e2e(i):
        brl[0] = tree.brlen[0] * (1.0 + 1e-3 * ((i % 5) - 2))      # a branch-length probe, as an optimiser would send
        e.set_model(0, md)                                          # eigensystem host -> device
        e.set_branch_lengths(0, brl)                                # host -> device
        if world == 1:
            return e.eval(want)[0][0]                               # log L (d1, d2) device -> host
        e.eval_device(want, out.data_ptr(), stream.cuda_stream)
        host_out.copy_(out, non_blocking=False)
        return float(host_out[0])

    for i in range(0 if a.profile else W):
        step_e2e(i)
    barrier()
    t0 = time.perf_counter()
    ev0.record(stream)
    for i in range(0 if a.profile else K):
        step_e2e(i)
    ev1.record(stream)
    barrier()
    e2e_ms = max(ev0.elapsed_time(ev1), 1e3 * (time.perf_counter() - t0))
    tms = torch.tensor([e2e_ms], dtype=torch.float64, device=device)
    if world > 1:
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
    e2e_ms = float(tms.item())
    log("[rank %d] e2e region done: %.3f ms/step" % (rank, e2e_ms / K))
    e.set_branch_lengths(0, tree.brlen)

    upd_step = tree.n_internal * w["patterns"] * w["C"] * w["S"]         # whole job (all shards)
    value = upd_step * K / (ms * 1e-3)
    # FP64 ceilings of this GPU, measured now, while the clock sampler of the timed region is still running
    dfma_peak, dmma_peak = capi.measure_fp64_peak(local) if rank == 0 else (None, None)
    clocks = sampler.stop() if rank == 0 else None

    # ---- the weak-scaling job of the same run (every GPU gets the workload's full pattern count) -------------------
    weak = None
    if world > 1 and a.scaling == "strong" and not a.profile and not a.no_weak:
        e.close()
        e = None
        ww = dict(w, patterns=w["patterns"] * world)
        t2, es2, r2, p2, codes2 = build_inputs(ww, rank, world, device)
        e, md = make_engine(ww, t2, es2, r2, p2, codes2, local, flags)
        shard.join_engine(e, device)
        for _ in range(W):
            step_device()
        barrier()
        ev0.record(stream)
        for _ in range(K):
            step_device()
        ev1.record(stream)
        barrier()
        tmsw = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.float64, device=device)
        dist.all_reduce(tmsw, op=dist.ReduceOp.MAX)
        wms = float(tmsw.item())
        weak = {"value": tree.n_internal * ww["patterns"] * w["C"] * w["S"] * K / (wms * 1e-3), "unit": "CLV updates/s",
                "ms_per_step": wms / K, "patterns": ww["patterns"], "patterns_per_gpu": w["patterns"], "lnl": float(out[0].item())}
        del codes2

    line = None
    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except OSError:
            pass
        hbm_peak = peaks.get("hbm_gbs", 6650.0)
        n_local = codes.shape[1]
        alg = algorithmic_bytes(tree, n_local, w["C"], w["S"])
        kms = st["prune_ms_sum"] / max(1, st["prune_count"])
        w4c = st["path"] == 1 and not w["derivs"] and os.environ.get("BPPGPU_WALK4C", "1") != "0"
        kname = {1: "walk4c_kernel" if w4c else "walk4_kernel", 2: "walkS_kernel", 3: "generic_node_kernel", 4: "dmma_node_kernel"}.get(st["path"], "?")
        fam20 = st["path"] == 4 and w["S"] == 20 and w["C"] <= 4 and os.environ.get("BPPGPU_FAMILY", "1") != "0"
        if fam20 or (st["path"] == 4 and w["S"] == 64 and w["C"] == 1 and os.environ.get("BPPGPU_FAMILY", "1") != "0"):
            kname = "dmma_prune_kernel"
        fp64_src = "measured in this run with bppgpu_measure_fp64_peak, under the clocks recorded in `clocks` (MEASURED_PEAKS.json has no FP64 figure)"
        rows = n_local * w["C"]
        if st["path"] == 4 and w["S"] >= 32:
            # dense contraction on the FP64 tensor cores (mma.sync DMMA; tcgen05 has no f64 kind).  frac = the DMMAs actually
            # issued (tip sons are table gathers) over the measured DMMA peak
            alg_flops = sum((2 * w["S"] * len(tree.sons(n)) + len(tree.sons(n)) - 1) * w["S"] for n in range(tree.nn)
                            if len(tree.sons(n))) * rows                  # SURVEY 8d: every son contracted, tips included
            exe_flops = flops_per_eval(tree, rows, w["S"])                # DMMA flops issued
            ach = exe_flops / (kms * 1e-3) / 1e12 if kms > 0 else None
            roofline = {"bound": "tensor", "kernel": kname + " (one launch per node; all launches of an evaluation timed together)",
                        "achieved": ach, "peak": dmma_peak, "unit": "TFLOP/s", "frac": ach / dmma_peak if ach else None,
                        "traffic": ncu_traffic_per_eval(a.workload, kname) if (not a.patterns and world == 1) else None,
                        "kernel_ms": kms, "launches_timed": st["prune_count"], "executed_dmma_flops_per_eval": exe_flops,
                        "algorithmic_flops_per_eval": alg_flops,
                        "algorithmic_tflops": alg_flops / (kms * 1e-3) / 1e12 if kms > 0 else None,
                        "peak_source": "FP64 mma.sync m8n8k4 " + fp64_src,
                        "note": "achieved = DMMA flops ISSUED per evaluation / pruning time (tip sons are table gathers and issue none); "
                                "algorithmic_flops counts (2 S k + k - 1) per CLV element with k sons as the reference does (SURVEY 8d)"}
        elif st["path"] == 1:
            # DNA register walk: every CLV stays on chip, HBM sees the tip codes only, the binding pipe is FP64 (CUDA cores)
            S = w["S"]
            fl = 0
            for n in range(tree.nn):
                sons = tree.sons(n)
                if len(sons):
                    fl += int((~tree.is_leaf[sons]).sum()) * (2 * S * S - S) + (len(sons) - 1) * S
            exe_flops = fl * rows
            ach = exe_flops / (kms * 1e-3) / 1e12 if kms > 0 else None
            traffic = ncu_traffic(kname) if (a.workload == DEFAULT and not a.patterns and world == 1) else None
            roofline = {"bound": "fp64", "kernel": kname, "achieved": ach, "peak": dfma_peak, "unit": "TFLOP/s",
                        "frac": ach / dfma_peak if ach else None, "traffic": traffic, "kernel_ms": kms,
                        "launches_timed": st["prune_count"], "executed_flops_per_launch": exe_flops,
                        "peak_source": "DFMA (CUDA-core FP64 pipe) " + fp64_src,
                        "hbm": {"bytes_moved_per_launch": traffic, "tip_code_bytes": int(tree.n_leaves) * n_local,
                                "achieved_gbs": traffic / (kms * 1e-3) / 1e9 if traffic and kms > 0 else None, "peak_gbs": hbm_peak,
                                "frac": traffic / (kms * 1e-3) / 1e9 / hbm_peak if traffic and kms > 0 else None},
                        "vs_level_scheduled": {"algorithmic_bytes_per_launch": alg, "hbm_floor_ms": alg / (hbm_peak * 1e9) * 1e3,
                                               "speedup_over_floor": alg / (hbm_peak * 1e9) * 1e3 / kms if kms > 0 else None,
                                               "note": "time a perfect level-scheduled kernel needs to stream 8*(1+internal sons) bytes per "
                                                       "CLV element (SURVEY 8d) at the measured HBM peak; this kernel does not move them"},
                        "note": "executed flops = (2 S^2 - S) per internal son + S per extra son, per (pattern, class) row: the DFMA/DMUL "
                                "the walk issues; CLVs never leave the SM, so the HBM roofline does not bound this kernel"}
        else:
            achieved = alg / (kms * 1e-3) / 1e9 if kms > 0 else None
            roofline = {"bound": "hbm", "kernel": kname, "achieved": achieved, "peak": hbm_peak, "unit": "GB/s",
                        "frac": achieved / hbm_peak if achieved else None,
                        "traffic": ncu_traffic_per_eval(a.workload, kname) if (not a.patterns and world == 1) else None,
                        "kernel_ms": kms,
                        "launches_timed": st["prune_count"], "algorithmic_bytes_per_launch": alg,
                        "peak_source": "MEASURED_PEAKS.json hbm_gbs (measured)" if peaks else "fallback 6650 GB/s",
                        "note": "algorithmic bytes = 8*(1+internal sons) per CLV element (SURVEY 8d); one launch per node, all "
                                "launches of an evaluation timed together"}
        if fam20 and w["derivs"]:
            # second kernel family of this workload: the per-father upper + d1/d2 pass, bound by the FP64 tensor pipe
            dms = ms / K - kms - st["pt_ms_sum"] / max(1, K)
            fl = family_dmma_flops(tree, n_local * w["C"])
            roofline["derivative_pass"] = {
                "kernel": "dmma_family_kernel (one launch per father)", "bound": "tensor", "ms": dms,
                "executed_dmma_flops": fl, "achieved": fl / (dms * 1e-3) / 1e12 if dms > 0 else None, "peak": dmma_peak,
                "unit": "TFLOP/s", "frac": fl / (dms * 1e-3) / 1e12 / dmma_peak if dms > 0 else None,
                "traffic": ncu_traffic_per_eval(a.workload, "dmma_family_kernel") if (not a.patterns and world == 1) else None,
                "note": "ms = step - pruning - P(t) (event timed); flops = DMMAs issued x 512"}
        line = {"metric": metric, "value": value, "unit": "CLV updates/s", "n_gpus": world, "steps": K, "warmup": W,
                "ms_per_step": ms / K, "higher_is_better": True, "scaling": a.scaling, "vs_baseline": None, "dtype": "f64",
                "data": "synthetic (tips simulated down a random tree under the model; every site kept as a pattern, weight 1)",
                "config": config, "logl_evals_per_s": K / (ms * 1e-3), "lnl": lnl_dev,
                "e2e": {"value": upd_step * K / (e2e_ms * 1e-3), "unit": "CLV updates/s", "h2d_bytes_per_step": h2d,
                        "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms / K,
                        "call": "bppgpu_set_model + bppgpu_set_branch_lengths + bppgpu_eval (host buffers)"},
                "gpu_launches": int(st["kernel_launches"]) * K, "launches_per_step": int(st["kernel_launches"]),
                "roofline": roofline, "clocks": clocks, "fp64_peaks_measured": {"dfma_tflops": dfma_peak, "dmma_m8n8k4_tflops": dmma_peak},
                "hbm_resident_bytes": int(st["hbm_bytes_resident"])}
        if weak is not None:
            line["weak"] = weak
        if world == 1 and not a.no_cpu:
            t0 = time.time()
            cb, sub, parity = cpu_leg(w, tree, es, rates, probs, codes, lnl_dev)
            # the same sample through the CUDA path: the checker, not the thing measured
            e2, _ = make_engine(w, tree, es, rates, probs, sub, local, flags)
            r2 = e2.eval(want)
            e2.close()
            cb["gpu_lnl_same_sample"] = float(r2[0][0])
            cb["rel_diff_vs_gpu"] = abs(r2[0][0] - cb["lnl_sample"]) / abs(cb["lnl_sample"])
            parity["rel_diff_sample"] = cb["rel_diff_vs_gpu"]
            line["cpu_baseline"] = cb
            line["parity"] = parity
            log("cpu leg %.1fs" % (time.time() - t0))
        emit(line)
        log("[rank 0] JSON line printed")
    e.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    try:
        rc = main()
    except BaseException:
        import traceback
        traceback.print_exc()
        sys.stderr.flush()
        raise
    sys.stdout.flush()
    sys.exit(rc)
