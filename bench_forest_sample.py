"""Forest sum and sample benchmark (cml_forests_sample / k_forest_sample, k_forest_sample_paths): prints ONE JSON line.

Workload: bench_forest_kbest.py's: 100,000 synth.make_forests forests of about 500 hyperedges each (52.4 M hyperedges),
fp64 weights drawn once (seeded).  Per n in {0, 1, 10, 100} (n = 0: totals only): the time of the synchronising
cml_forests_sample call (host clock, median of the repeats, after a warm-up call), the time of its kernels (CUDA
events: the host levelisation and the copies are the rest of the call), samples/s per call, hyperedges/s over kernel
time, scratch bytes and chunks.  n = 1 and 10 return the node lists; at n = 100 the call asks for weights and sizes
only (the node lists of 10 million samples would not fit the host).  cml_forests_viterbi (k_forest_viterbi) is timed
too, alternating with cml_forests_sample in the same process.
Parity: cml_forests_sample against the CPU reference (tests/forest_sample_helpers.py: memoised inside recursion and a
recursive walk per sample) on the first 40 forests at n = 10, under the comparison rule there; the line reports
parity = false when any check fails.  The GPU's name, power limit and max SM clock come from nvidia-smi.

  python bench_forest_sample.py [--repeats R] [--forests N]
It writes nothing to disk.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
NS = (0, 1, 10, 100)
PARITY_FORESTS, PARITY_N = 40, 10
NODES_UP_TO_N = 10
SEED = 20290101


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--forests", type=int, default=100000)
    a = ap.parse_args()
    import numpy as np
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_forest_sample.py needs a CUDA device (there is no CPU fallback)")
    from bench_kbest import gpu_facts
    from carmel_b200 import synth
    from carmel_b200.forest_api import Forests
    t0 = time.perf_counter()
    fs = synth.make_forests(n_forests=a.forests, templates=0)
    arrays = (fs["node_off"], fs["next"], fs["label"], fs["backref"])
    f = Forests(0, 64)
    f.set_rules(fs["rulespace"], fs["group_off"], fs["group_members"])
    ln_w = np.log(np.random.default_rng(20271801).uniform(0.01, 1.0, fs["rulespace"]))
    f.set_params(ln_w)
    f.normalize_params()
    ln_w = f.get_params()
    res = {"bench": "forest_sample", "gpu": gpu_facts(), "repeats": a.repeats, "forests": a.forests,
           "nodes": fs["nodes"], "hyperedges": fs["hyperedges"], "setup_s": time.perf_counter() - t0, "n": {}}
    med = lambda xs: sorted(xs)[len(xs) // 2]

    def sample(n):
        lnw, _, _, _, total = f.sample(n, SEED, *arrays, nodes=n <= NODES_UP_TO_N)
        st = f.sample_stats()
        st["samples"] = int((lnw > -math.inf).sum())
        st["forests_with_derivation"] = int((total > -math.inf).sum())
        return st

    f.viterbi(*arrays)  # warm-up
    tv_all = []
    for n in NS:
        sample(n)  # warm-up
        ts, ms, tv = [], [], []
        for _ in range(a.repeats):
            t1 = time.perf_counter()
            st = sample(n)
            ts.append(time.perf_counter() - t1)
            ms.append(st["kernel_ms"])
            t1 = time.perf_counter()
            f.viterbi(*arrays)
            tv.append(time.perf_counter() - t1)
        tv_all += tv
        t_call, t_kernel = med(ts), med(ms)
        res["n"][str(n)] = {"call_s": t_call, "kernel_ms": t_kernel, "host_and_copies_s": t_call - t_kernel * 1e-3,
                            "nodes_returned": 0 < n <= NODES_UP_TO_N, "samples": st["samples"],
                            "forests_with_derivation": st["forests_with_derivation"],
                            "samples_per_s_call": st["samples"] / t_call,
                            "hyperedges_per_s_kernel": fs["hyperedges"] / (t_kernel * 1e-3) if t_kernel > 0 else None,
                            "scratch_bytes": st["scratch_bytes"], "chunks": st["chunks"], "viterbi_call_s": med(tv)}
    res["viterbi"] = {"call_s": med(tv_all),
                      "note": "k_forest_viterbi has no kernel timer: a whole synchronising call, alternated with the sampler"}
    # parity on the first forests
    from forest_sample_helpers import EXEMPT_SHARE, compare_samples, forest_samplers
    n = PARITY_FORESTS
    sub = (fs["node_off"][:n + 1], fs["next"][:int(fs["node_off"][n])], fs["label"][:int(fs["node_off"][n])],
           fs["backref"][:int(fs["node_off"][n])])
    par = {"forests": n, "n": PARITY_N, "ok": False}
    try:
        lnw, n_and, base, nodes, total = f.sample(PARITY_N, SEED, *sub)
        n_ex = 0
        for i, s in enumerate(forest_samplers(*sub, ln_w)):
            got = [(float(lnw[i, r]), tuple(int(x) for x in nodes[int(base[i * PARITY_N + r]):][:int(n_and[i, r])]))
                   for r in range(PARITY_N)]
            n_ex += compare_samples(s, s.draw(SEED, i, PARITY_N), float(total[i]), got)
        assert n_ex <= EXEMPT_SHARE * PARITY_N * n, n_ex
        par["exempt"] = n_ex
        par["ok"] = True
    except AssertionError as ex:
        par["failure"] = repr(ex)[:400]
    res["parity_detail"] = par
    res["parity"] = par["ok"]
    print(json.dumps(res))


if __name__ == "__main__":
    main()
