"""k-best decode benchmark (cml_kbest / k_kbest): prints ONE JSON line.

Workloads (lattice path, fp64 log space, layered CSR: the layout the decode needs):
  cipher  configs[1]: synth.write_cipher, 2,000 lines x 50, 27x27 channel o letter-bigram LM
  hmm     a configs[2] subset: synth.write_hmm, 100,000 sentences (32 tags, 5k vocab, 4 tags/word)
Per workload and k in {1, 10, 100}: the time of the synchronising cml_kbest call (host clock, median of the repeats,
after a warm-up call), the time of its derivation kernels (CUDA events), derivations/s and lattice arcs/s, scratch
bytes and chunks.  At k = 1 the same is reported for cml_viterbi, alternating with cml_kbest in the same process.
Parity: cml_kbest against the CPU reference (tests/kbest_helpers.py: a lazy enumeration over the lattices the CPU
oracle builds) on the first 40 lines at k = 10, under the comparison rule there; the line reports parity = false when any
check fails.  The CPU baseline is that reference's rate on the sample (one Python process, lattices already built).
The GPU's name, power limit and max SM clock come from nvidia-smi.

  python bench_kbest.py [--repeats R] [--hmm-sentences N]
Everything it writes goes to a temporary directory.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "tests"))
ORACLE = os.path.join(ROOT, "oracle", "_build", "carmel_oracle")
KS = (1, 10, 100)
PARITY_LINES, PARITY_K = 40, 10
JOB_FLAGS = ["--no-ell", "--no-dense", "--no-lane"]


def gpu_facts():
    q = "name,power.limit,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=60).stdout.strip().splitlines()[0]
        return dict(zip(("name", "power_limit", "max_sm_clock"), (x.strip() for x in out.split(","))))
    except Exception as ex:  # the numbers below still stand, without the card's facts
        return {"error": str(ex)}


def timed(fn, repeats):
    fn()  # warm-up: module load, allocations
    ts, ms = [], []
    for _ in range(repeats):
        t0 = time.perf_counter()
        stats = fn()
        ts.append(time.perf_counter() - t0)
        ms.append(stats["kernel_ms"])
    ts.sort()
    ms.sort()
    return ts[len(ts) // 2], ms[len(ms) // 2], stats


def parity(w, tmp):
    """GPU (cml_kbest through a Job on the first PARITY_LINES lines) vs the CPU reference at k = PARITY_K"""
    from carmel_b200 import Job, synth
    from helpers import read_estimate_dump, read_trellis_dump
    from kbest_helpers import Lattices, compare_kbest
    data = os.path.join(tmp, f"{w['workload']}.head.data")
    synth.head_corpus(w["files"][0], data, PARITY_LINES)
    args = [w["argv"][0], data, *w["files"][1:]]
    subprocess.run([ORACLE, f"--dump-trellis={tmp}/o.t", f"--dump-estimate={tmp}/o.e", *args], check=True,
                   capture_output=True)
    lat = Lattices(read_trellis_dump(f"{tmp}/o.t"), read_estimate_dump(f"{tmp}/o.e")["ln_w"])
    t0 = time.perf_counter()
    want = [lat.kbest(e, PARITY_K) for e in range(lat.t["n_ex"])]
    t_ref = time.perf_counter() - t0
    job = Job([*JOB_FLAGS, *args])
    ctx = job.prepare()
    lnw, plen, base, arcs = ctx.kbest(PARITY_K)
    res = {"lines": PARITY_LINES, "k": PARITY_K, "examples": len(want), "ok": False}
    try:
        assert lnw.shape[0] == len(want) == PARITY_LINES, (lnw.shape, len(want))
        for e in range(len(want)):
            got = []
            for r in range(PARITY_K):
                i = e * PARITY_K + r
                got.append((float(lnw[e, r]), tuple(int(x) for x in arcs[base[i]:base[i] + plen[e, r]])))
            compare_kbest(want[e], got, lambda p, e=e: lat.weight(e, p))
        res["ok"] = True
    except AssertionError as ex:
        res["failure"] = repr(ex)[:400]
    job.close()
    n_der = sum(1 for ex in want for wt, _ in ex if wt > -math.inf)
    res["cpu_reference"] = {"seconds": t_ref, "derivations": n_der, "derivations_per_s": n_der / t_ref,
                            "note": "the Python lazy enumeration of tests/kbest_helpers.py, one process, lattices built"}
    return res


def run_workload(w, repeats, tmp):
    from carmel_b200 import Job
    t0 = time.perf_counter()
    job = Job([*JOB_FLAGS, *w["argv"]])
    ctx = job.prepare()
    tot = ctx.trellis_totals()
    out = {"examples": tot["examples"], "lattice_states": tot["states"], "lattice_arcs": tot["arcs"],
           "lattice_levels": tot["levels"], "prepare_s": time.perf_counter() - t0, "k": {}}

    def kbest(k):
        lnw, _, _, _ = ctx.kbest(k)
        st = ctx.kbest_stats()
        st["derivations"] = int((lnw > -math.inf).sum())
        return st

    def viterbi():
        lnw, _, _, _ = ctx.viterbi()
        st = ctx.kbest_stats()
        st["derivations"] = int((lnw > -math.inf).sum())
        return st

    for k in KS:
        if k == 1:  # alternate the two 1-best implementations
            ctx.kbest(1), ctx.viterbi()
            tk, tv, mk, mv = [], [], [], []
            for _ in range(repeats):
                for fn, ts, ms in ((kbest, tk, mk), (viterbi, tv, mv)):
                    t0 = time.perf_counter()
                    st = fn(1) if fn is kbest else fn()
                    ts.append(time.perf_counter() - t0)
                    ms.append(st["kernel_ms"])
            med = lambda xs: sorted(xs)[len(xs) // 2]
            st = kbest(1)
            t_call, t_kernel = med(tk), med(mk)
            out["viterbi_k1"] = {"call_s": med(tv), "kernel_ms": med(mv),
                                 "kbest_over_viterbi_kernel": med(mk) / max(med(mv), 1e-9)}
        else:
            t_call, t_kernel, st = timed(lambda: kbest(k), repeats)
        out["k"][str(k)] = {"call_s": t_call, "kernel_ms": t_kernel, "derivations": st["derivations"],
                            "derivations_per_s_call": st["derivations"] / t_call,
                            "lattice_arcs_per_s_kernel": tot["arcs"] / (t_kernel * 1e-3) if t_kernel > 0 else None,
                            "scratch_bytes": st["scratch_bytes"], "chunks": st["chunks"]}
    job.close()
    out["parity"] = parity(w, tmp)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--hmm-sentences", type=int, default=100000)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_kbest.py needs a CUDA device (there is no CPU fallback)")
    from carmel_b200 import synth
    global ORACLE
    res = {"bench": "kbest", "gpu": gpu_facts(), "repeats": a.repeats, "workloads": {}}
    with tempfile.TemporaryDirectory() as tmp:
        if not os.path.exists(ORACLE):  # a tree built without the oracle: build it in the temporary directory
            subprocess.run(["make", "-C", os.path.join(ROOT, "oracle"), f"OUT={tmp}/oracle", f"{tmp}/oracle/carmel_oracle"],
                           check=True, capture_output=True)
            ORACLE = os.path.join(tmp, "oracle", "carmel_oracle")
        for name, mk in (("cipher", lambda d: synth.write_cipher(d, n_lines=2000, line_len=50)),
                         ("hmm", lambda d: synth.write_hmm(d, n_sent=a.hmm_sentences))):
            d = os.path.join(tmp, name)
            w = mk(d)
            res["workloads"][name] = run_workload(w, a.repeats, d)
    res["parity"] = all(v["parity"]["ok"] for v in res["workloads"].values())
    print(json.dumps(res))


if __name__ == "__main__":
    main()
