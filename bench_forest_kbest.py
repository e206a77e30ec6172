"""Forest k-best decode benchmark (cml_forests_kbest / k_forest_kbest): prints ONE JSON line.

Workload: the configs[4] shape from synth.make_forests: 100,000 forests of about 500 hyperedges each, fp64 weights
drawn once (seeded).  Per k in {1, 10, 100}: the time of the synchronising cml_forests_kbest call (host clock, median of
the repeats, after a warm-up call), the time of its derivation kernels (CUDA events), derivations/s, hyperedges/s
(kernel), scratch bytes and chunks.  At k = 100 the call asks for scores and sizes only (the node lists of 10 million
derivations would not fit the host); k = 1 and 10 return the node lists.  At k = 1, cml_forests_viterbi (k_forest_viterbi)
is timed too, alternating with cml_forests_kbest in the same process.
Parity: cml_forests_kbest against the CPU reference (tests/forest_kbest_helpers.py: a lazy enumeration with a candidate
heap per node) on the first 40 forests at k = 10, under the comparison rule there; the line reports parity = false when
any check fails.  The GPU's name, power limit and max SM clock come from nvidia-smi.

  python bench_forest_kbest.py [--repeats R] [--forests N]
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
KS = (1, 10, 100)
PARITY_FORESTS, PARITY_K = 40, 10
NODES_UP_TO_K = 10


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--forests", type=int, default=100000)
    a = ap.parse_args()
    import numpy as np
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_forest_kbest.py needs a CUDA device (there is no CPU fallback)")
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
    res = {"bench": "forest_kbest", "gpu": gpu_facts(), "repeats": a.repeats, "forests": a.forests,
           "nodes": fs["nodes"], "hyperedges": fs["hyperedges"], "setup_s": time.perf_counter() - t0, "k": {}}
    med = lambda xs: sorted(xs)[len(xs) // 2]

    def kbest(k):
        score, _, _, _ = f.kbest(k, *arrays, nodes=k <= NODES_UP_TO_K)
        st = f.kbest_stats()
        st["derivations"] = int((score > -math.inf).sum())
        return st

    for k in KS:
        kbest(k)  # warm-up
        tk, mk, tv = [], [], []
        for _ in range(a.repeats):
            t1 = time.perf_counter()
            st = kbest(k)
            tk.append(time.perf_counter() - t1)
            mk.append(st["kernel_ms"])
            if k == 1:
                t1 = time.perf_counter()
                f.viterbi(*arrays)
                tv.append(time.perf_counter() - t1)
        t_call, t_kernel = med(tk), med(mk)
        res["k"][str(k)] = {"call_s": t_call, "kernel_ms": t_kernel, "nodes_returned": k <= NODES_UP_TO_K,
                            "derivations": st["derivations"], "derivations_per_s_call": st["derivations"] / t_call,
                            "hyperedges_per_s_kernel": fs["hyperedges"] / (t_kernel * 1e-3) if t_kernel > 0 else None,
                            "scratch_bytes": st["scratch_bytes"], "chunks": st["chunks"]}
        if k == 1:
            res["viterbi_k1"] = {"call_s": med(tv), "kbest_over_viterbi_call": t_call / max(med(tv), 1e-9),
                                 "note": "k_forest_viterbi has no kernel timer: both are whole synchronising calls"}
    # parity on the first forests
    from forest_kbest_helpers import compare_kbest, forest_refs
    n = PARITY_FORESTS
    sub = (fs["node_off"][:n + 1], fs["next"][:int(fs["node_off"][n])], fs["label"][:int(fs["node_off"][n])],
           fs["backref"][:int(fs["node_off"][n])])
    par = {"forests": n, "k": PARITY_K, "ok": False}
    try:
        score, n_and, base, nodes = f.kbest(PARITY_K, *sub)
        for i, ref in enumerate(forest_refs(*sub, ln_w)):
            got = [(float(score[i, r]), tuple(int(x) for x in nodes[int(base[i * PARITY_K + r]):][:int(n_and[i, r])]))
                   for r in range(PARITY_K)]
            compare_kbest(ref.kbest(PARITY_K), got, ref.score_of)
        par["ok"] = True
    except AssertionError as ex:
        par["failure"] = repr(ex)[:400]
    res["parity_detail"] = par
    res["parity"] = par["ok"]
    print(json.dumps(res))


if __name__ == "__main__":
    main()
