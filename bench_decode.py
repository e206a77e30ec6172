"""Benchmark of decoding new strings with the other tape free (cml_build_free_trellises / k_build_free, then
cml_add_trellises and cml_viterbi / cml_kbest; carmel-b200 --decode): prints ONE JSON line.

Workloads (both have a real free tape):
  decipherment  a 27-letter bigram LM written as an FSA with b:b arcs (the plaintext on the input tape) o the 27 x 27
                channel of synth.write_cipher; 2,000 cipher lines of 50 decoded with the output tape given
  tagging       the configs[2] shape of synth.write_hmm with a tag:tag bigram, so the tags are the free input; 100,000
                sentences decoded with the output tape given
The calls are timed in ONE process through the ctypes Context, on the composed machine and the normalised arc weights
the command line decodes with (the CPU oracle's --write-composed / --dump-estimate: the same arc table, the same
weights).  Per workload and k in {1, 10}: one warm-up round, then the medians of R rounds of
  - the builder call (cml_build_free_trellises' own wall time) and its k_build_free kernels (CUDA events),
  - cml_add_trellises (host clock; host code: the layered-CSR flattening and upload),
  - the decode call (cml_viterbi for k = 1, cml_kbest otherwise; host clock) and its kernels (cml_kbest_stats),
  - lattice arcs/s of the builder kernels.
Strings/s end to end is the whole command (`carmel-b200 --decode`: reading and composing the model, building, decoding,
writing the file; a warm-up run, then the median of R runs).  Parity: the command line's file for the first 40 strings at
k = 10 against the CPU reference (tests/decode_helpers.py) under the comparison rule of tests/kbest_helpers.py; the CPU
reference's lattice build time on those 40 strings is reported beside it.  The GPU's name, power limit and max SM clock
come from nvidia-smi.

  python bench_decode.py [--repeats R] [--tagging-sentences N]
Everything it writes goes to a temporary directory.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import re
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
ORACLE = os.path.join(ROOT, "oracle", "_build", "carmel_oracle")
KS = (1, 10)
PARITY_LINES, PARITY_K = 40, 10


def gpu_facts():
    q = "name,power.limit,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=60).stdout.strip().splitlines()[0]
        return dict(zip(("name", "power_limit", "max_sm_clock"), (x.strip() for x in out.split(","))))
    except Exception as ex:  # the numbers below still stand, without the card's facts
        return {"error": str(ex)}


def free_input(path):
    """the LM / tag bigram with each *e*:x arc made x:x, so its symbols are on the composed machine's input tape"""
    text = open(path).read()
    open(path, "w").write(re.sub(r'\*e\* ("[^"]*")', r"\1 \1", text))


def copy_lines(src, dst, start=0, step=1, n=None):
    """lines start, start + step, ... of src (at most n) -> dst; returns them"""
    lines = open(src).read().splitlines()[start::step][:n]
    open(dst, "w").write("\n".join(lines) + "\n")
    return lines


def med(xs):
    return sorted(xs)[len(xs) // 2]


def cli_wall(model, strings, out, k):
    from carmel_b200 import CLI_PATH
    t0 = time.perf_counter()
    p = subprocess.run([CLI_PATH, f"--decode={out}", "--given=output", "-k", str(k), strings, *model],
                       capture_output=True, text=True)
    wall = time.perf_counter() - t0
    assert p.returncode == 0, p.stderr[-2000:]
    return wall


def in_process(m, lines, repeats):
    """the builder, cml_add_trellises and the decoders in one process, warm"""
    from carmel_b200 import api as cb
    import decode_helpers as D
    ids = [D.symbols(ln, m["alphabet"]) for ln in lines]
    off = np.zeros(len(ids) + 1, np.uint64)
    off[1:] = np.cumsum([len(x) for x in ids])
    sym = np.fromiter((s for x in ids for s in x), np.uint32, int(off[-1]))
    ctx = cb.Context(precision=64, space=cb.SPACE_LOG)
    ctx.set_option(cb.OPT_NO_ELL, 1)
    ctx.set_trivial_model(m["arc_in"].size)
    ctx.set_params(m["ln_w"])
    keys = ("ex_states", "ex_fin", "ex_weight", "arc_off", "arc_dst", "arc_id")
    res = {}
    for k in KS:
        def round_():
            b = ctx.build_free_trellises(m, (off, sym), 1)
            ctx.clear_trellises()
            t0 = time.perf_counter()
            ctx.add_trellises(*(b[x] for x in keys))
            t_add = time.perf_counter() - t0
            t0 = time.perf_counter()
            lnw = (ctx.kbest(k) if k > 1 else ctx.viterbi())[0]
            t_dec = time.perf_counter() - t0
            st = ctx.kbest_stats()
            return dict(build_s=b["stats"]["seconds"], build_kernel_ms=b["stats"]["kernel_ms"], chunks=b["stats"]["chunks"],
                        lattices=b["n_ex"], lattice_states=int(b["ex_states"].sum()), lattice_arcs=int(b["arc_id"].size),
                        add_trellises_s=t_add, decode_s=t_dec, decode_kernel_ms=st["kernel_ms"],
                        derivations=int((lnw > -math.inf).sum()))
        round_()  # warm-up: module loads, allocations
        runs = [round_() for _ in range(repeats)]
        r = {key: med([x[key] for x in runs]) for key in runs[0]}
        r["lattice_arcs_per_s_build_kernel"] = r["lattice_arcs"] / (r["build_kernel_ms"] * 1e-3)
        res[str(k)] = r
    ctx.close()
    return res


def parity(m, model, strings, tmp):
    import decode_helpers as D
    from kbest_helpers import compare_kbest
    head = os.path.join(tmp, "head.txt")
    lines = copy_lines(strings, head, n=PARITY_LINES)
    out = os.path.join(tmp, "head.out")
    cli_wall(model, head, out, PARITY_K)
    ids = [D.symbols(ln, m["alphabet"]) for ln in lines]
    t0 = time.perf_counter()
    lat = D.free_lattices(m, ids, 1)
    t_build = time.perf_counter() - t0
    want, _, L = D.reference_kbest(m, ids, 1, PARITY_K, lat)
    got = D.read_decode(out, PARITY_K)
    res = {"strings": len(lines), "k": PARITY_K, "ok": False, "cpu_reference_build_s": t_build,
           "cpu_reference_lattice_arcs": int(lat["arc_id"].size),
           "note": "the CPU reference build is the Python restatement of tests/decode_helpers.py, one process"}
    try:
        assert len(got) == len(want) == len(lines)
        lat_of = {int(e): i for i, e in enumerate(lat["kept"])}
        for e in range(len(lines)):
            wo = (lambda p, i=lat_of[e]: L.weight(i, p)) if e in lat_of else (lambda p: None)
            compare_kbest([x[:2] for x in want[e]], [x[:2] for x in got[e]], wo)
            for w, p, s in got[e]:
                assert w == -math.inf or s == D.decoded_string(m, p, 1), (e, s)
        res["ok"] = True
    except AssertionError as ex:
        res["failure"] = repr(ex)[:400]
    return res


def run_workload(model, strings, repeats, tmp):
    import decode_helpers as D
    m = D.reference_model(ORACLE, tmp, model)
    lines = open(strings).read().splitlines()
    res = {"strings": len(lines), "composed_arcs": int(m["arc_in"].size), "k": in_process(m, lines, repeats)}
    for k in KS:
        out = os.path.join(tmp, f"k{k}.out")
        cli_wall(model, strings, out, k)  # warm-up (file cache)
        wall = med([cli_wall(model, strings, out, k) for _ in range(repeats)])
        res["k"][str(k)].update(cli_wall_s=wall, strings_per_s_end_to_end=len(lines) / wall)
    res["parity"] = parity(m, model, strings, tmp)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--tagging-sentences", type=int, default=100000)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_decode.py needs a CUDA device (there is no CPU fallback)")
    from carmel_b200 import synth
    global ORACLE
    res = {"bench": "decode", "gpu": gpu_facts(), "repeats": a.repeats, "workloads": {}}
    with tempfile.TemporaryDirectory() as tmp:
        if not os.path.exists(ORACLE):  # a tree built without the oracle: build it in the temporary directory
            subprocess.run(["make", "-C", os.path.join(ROOT, "oracle"), f"OUT={tmp}/oracle", f"{tmp}/oracle/carmel_oracle"],
                           check=True, capture_output=True)
            ORACLE = os.path.join(tmp, "oracle", "carmel_oracle")
        for name, mk in (("decipherment", lambda d: synth.write_cipher(d, n_lines=2000, line_len=50)),
                         ("tagging", lambda d: synth.write_hmm(d, n_sent=a.tagging_sentences))):
            d = os.path.join(tmp, name)
            w = mk(d)
            data, lm, channel = w["files"]
            free_input(lm)
            strings = os.path.join(d, "strings.txt")
            copy_lines(data, strings, start=1, step=2)  # the output lines of the pair corpus
            res["workloads"][name] = run_workload(["--train-cascade", lm, channel], strings, a.repeats, d)
    res["parity"] = all(v["parity"]["ok"] for v in res["workloads"].values())
    print(json.dumps(res))


if __name__ == "__main__":
    main()
