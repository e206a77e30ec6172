"""Sum and sample benchmark (cml_sample / k_sample): prints ONE JSON line.

Workloads: bench_kbest.py's two (lattice path, fp64 log space, layered CSR): the configs[1] cipher (2,000 lines x 50)
and 100,000 HMM sentences.  Per workload and n in {0, 1, 10, 100}: the time of the synchronising cml_sample call (host
clock, median of the repeats after a warm-up call), the time of its k_sample launches (CUDA events), samples/s of the
call and lattice arcs/s of the kernel (each arc is read once by the beta pass), scratch bytes and chunks.  cml_viterbi is
timed in the same process, alternating with cml_sample, for scale.  Parity: the first 40 lattices at n = 100 against the
CPU reference (tests/sample_helpers.py over the lattices the CPU oracle builds) under the comparison rule there, and
the ln totals to 1e-12; the line reports parity = false when any check fails.  The GPU's name, power limit and max SM
clock come from nvidia-smi in the same run.

  python bench_sample.py [--repeats R] [--hmm-sentences N]
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
import bench_kbest as BK  # noqa: E402  (the workloads, flags and card facts)

NS = (0, 1, 10, 100)
PARITY_LINES, PARITY_N, SEED = 40, 100, 1


def parity(w, tmp, oracle):
    """cml_sample through a Job on the first PARITY_LINES lines vs the CPU reference"""
    from carmel_b200 import Job, synth
    from helpers import read_estimate_dump, read_trellis_dump
    from kbest_helpers import Lattices
    import sample_helpers as S
    data = os.path.join(tmp, f"{w['workload']}.head.data")
    synth.head_corpus(w["files"][0], data, PARITY_LINES)
    args = [w["argv"][0], data, *w["files"][1:]]
    subprocess.run([oracle, f"--dump-trellis={tmp}/o.t", f"--dump-estimate={tmp}/o.e", *args], check=True,
                   capture_output=True)
    smp = S.Sampler(Lattices(read_trellis_dump(f"{tmp}/o.t"), read_estimate_dump(f"{tmp}/o.e")["ln_w"]))
    job = Job([*BK.JOB_FLAGS, *args])
    ctx = job.prepare()
    tot, lnw, plen, base, arcs = ctx.sample(PARITY_N, SEED)
    res = {"lines": PARITY_LINES, "n": PARITY_N, "examples": int(tot.size), "ok": False, "exempt": 0}
    try:
        assert tot.size == PARITY_LINES, tot.size
        for e in range(tot.size):
            want = smp.ln_total(e)
            assert want == tot[e] or abs(want - tot[e]) <= 1e-12 * max(1.0, abs(want)), (e, want, tot[e])
            got = [(float(lnw[e, r]), tuple(int(x) for x in arcs[base[e * PARITY_N + r]:][:plen[e, r]]))
                   for r in range(PARITY_N)]
            res["exempt"] += S.compare_draws(smp.draw(e, SEED, e, PARITY_N), got)
        assert res["exempt"] <= 0.001 * PARITY_N * tot.size, res["exempt"]
        res["ok"] = True
    except AssertionError as ex:
        res["failure"] = repr(ex)[:400]
    job.close()
    return res


def run_workload(w, repeats, tmp, oracle):
    from carmel_b200 import Job
    t0 = time.perf_counter()
    job = Job([*BK.JOB_FLAGS, *w["argv"]])
    ctx = job.prepare()
    tot = ctx.trellis_totals()
    out = {"examples": tot["examples"], "lattice_states": tot["states"], "lattice_arcs": tot["arcs"],
           "lattice_levels": tot["levels"], "prepare_s": time.perf_counter() - t0, "n": {}}
    med = lambda xs: sorted(xs)[len(xs) // 2]
    for n in NS:
        ctx.sample(n, SEED), ctx.viterbi()  # warm-up
        ts, ms, tv, mv = [], [], [], []
        for _ in range(repeats):  # alternate cml_sample and cml_viterbi
            t0 = time.perf_counter()
            total = ctx.sample(n, SEED)[0]
            ts.append(time.perf_counter() - t0)
            st = ctx.sample_stats()
            ms.append(st["kernel_ms"])
            t0 = time.perf_counter()
            ctx.viterbi()
            tv.append(time.perf_counter() - t0)
            mv.append(ctx.kbest_stats()["kernel_ms"])
        t_call, t_kernel = med(ts), med(ms)
        drawn = n * int((total > -math.inf).sum())
        out["n"][str(n)] = {"call_s": t_call, "kernel_ms": t_kernel, "samples": drawn,
                            "samples_per_s_call": drawn / t_call if n else None,
                            "lattice_arcs_per_s_kernel": tot["arcs"] / (t_kernel * 1e-3) if t_kernel > 0 else None,
                            "scratch_bytes": st["scratch_bytes"], "chunks": st["chunks"],
                            "viterbi_call_s": med(tv), "viterbi_kernel_ms": med(mv)}
    job.close()
    out["parity"] = parity(w, tmp, oracle)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--hmm-sentences", type=int, default=100000)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_sample.py needs a CUDA device (there is no CPU fallback)")
    from carmel_b200 import synth
    res = {"bench": "sample", "gpu": BK.gpu_facts(), "repeats": a.repeats, "workloads": {}}
    oracle = BK.ORACLE
    with tempfile.TemporaryDirectory() as tmp:
        if not os.path.exists(oracle):  # a tree built without the oracle: build it in the temporary directory
            subprocess.run(["make", "-C", os.path.join(ROOT, "oracle"), f"OUT={tmp}/oracle", f"{tmp}/oracle/carmel_oracle"],
                           check=True, capture_output=True)
            oracle = os.path.join(tmp, "oracle", "carmel_oracle")
        for name, mk in (("cipher", lambda d: synth.write_cipher(d, n_lines=2000, line_len=50)),
                         ("hmm", lambda d: synth.write_hmm(d, n_sent=a.hmm_sentences))):
            d = os.path.join(tmp, name)
            w = mk(d)
            res["workloads"][name] = run_workload(w, a.repeats, d, oracle)
    res["parity"] = all(v["parity"]["ok"] for v in res["workloads"].values())
    print(json.dumps(res))


if __name__ == "__main__":
    main()
