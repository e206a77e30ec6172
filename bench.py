#!/usr/bin/env python
"""bench.py -- EM-iteration throughput of the B200-native carmel training path (trellis arcs/s).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--legs all|none|c2,c3,c5,c4,cli]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

ONE JSON line (rank 0).  A step = one EM iteration over resident derivation lattices: class / arc weights from the
parameter table, forward, fused backward + expected counts, all-reduce of the count table (NCCL, issued by the library on
its own stream when N > 1), normalisation M-step -- one C-ABI call (cml_em_step), one host synchronisation.

main line   BASELINE.json configs[1]: cipher decipherment, 100k letters per GPU (2000 lines x 50), on the LATTICE path
            (--no-dense): the sparse-trellis forward/backward kernel the >= 50% HBM target is about (k_fb_wide).
            Weak scaling (2000 lines per GPU).
  value       whole-job trellis arcs/s, lattices resident in HBM, CUDA events on the library's stream, max over ranks
  e2e         same metric through the C ABI with HOST buffers every step: parameters H2D from pinned memory; likelihood,
              expected counts and new parameters D2H
  roofline    the forward/backward/count kernel alone: algorithmic bytes (SURVEY.md 8d: 16 B/arc +
              2*sizeof(real)*states/arcs) / its CUDA-event time (events around the kernel on the launching stream,
              measured in a separate un-graphed pass of the same E-step), against MEASURED_PEAKS.json:hbm_gbs
  parity      per-example ln P of the GPU path against the CPU oracle on the cpu_baseline sample (fails above 1e-6 / 1e-4)
  parity_n    N > 1: rank 0 alone over the same total corpus: sum ln P and the reduced count table must agree to 1e-9
legs        dense_path (same corpus, the product's default dense-state path), c3 (configs[2] HMM, 1M sentences IN TOTAL,
            strong scaling, lattice path + dense-state path), c5 (configs[4] forests, 100k in total, every forest its own
            shape, strong scaling), c4 (configs[3] Gibbs, 1M letters, N = 1 only: the exact sampler is sequential),
            e2e_cli (wall time of `carmel-b200 --train-cascade -M 20` against the CPU oracle), tf32_peak (measured in-run)
cpu_baseline / --impl reference
            the CPU oracle (restatement of the reference algorithm; the reference binary needs Boost and cannot be built
            here) timed on this box's host cores on a bounded sample of the main workload.
--dump-outputs DIR
            after the main line's timed steps, rank 0 writes what the last timed EM iteration gave its caller as
            DIR/<name>.npy (float64): step_result (sum ln P, sum weighted ln P, examples without a derivation, max weight
            change), params (ln weights after the M-step), counts (the all-reduced expected counts), example_ln_p (ln P of
            rank 0's examples).  Inputs are seeded, so two builds can be compared output for output.  Above 64 MB in all,
            every array is cut to the same share by a fixed seeded choice of indices.
"""
from __future__ import annotations

import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ORACLE = os.path.join(ROOT, "oracle", "_build", "carmel_oracle")
FALLBACK_HBM_GBS = 6650.0  # /opt/skills/guides/B200_PROFILING.md fallback
METRIC, UNIT = "em_iteration_trellis_arcs_per_sec", "trellis arcs/s"
CIPHER_LINES, CIPHER_SAMPLE = 2000, 160
C3_SENTENCES, C3_SAMPLE = 1000000, 16000
DUMP_BYTES = (64 << 20) - (16 << 10)  # --dump-outputs: 64 MB in all, less room for the .npy headers


def measured_traffic(kernel, units=None):
    """dram bytes per launch of a kernel from the committed ncu captures (profiles/traffic.json), or None.  The capture
    names the units (arcs / positions / hyperedges) its launch processed: a launch over `units` units is charged
    bytes / captured units x units (same workload family at another size)."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get(kernel)
        if not t:
            return None
        if units and t.get("units"):
            return float(t["bytes"]) / float(t["units"]) * float(units)
        return float(t["bytes"])
    except Exception:
        return None


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)), "measured"
        except Exception:
            pass
    return {"hbm_gbs": FALLBACK_HBM_GBS}, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)"""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.rows = []
        self.p = None
        self.gpu = gpu_index

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "100", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.p = None

    def _read(self):
        for ln in self.p.stdout:
            self.rows.append([x.strip() for x in ln.split(",")])

    def stop(self):
        if self.p:
            time.sleep(0.15)
            self.p.terminate()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def main_config(world: int) -> dict:
    """config of the main line; the reference arm prints the same dict"""
    return {"workload": "configs[1] cipher decipherment: 27x27 channel o 27-state locked bigram LM, 100k-letter synthetic "
                        "ciphertext per GPU (2000 lines x 50), EM, f64 scaled space",
            "examples_per_gpu": CIPHER_LINES, "space": "scaled",
            "l2": "inputs larger than L2: 1.2 GB of lattice records streamed per iteration and GPU (L2 126 MB)",
            "parallelism": f"examples sharded over {world} GPU(s), one NCCL all-reduce of the count table per iteration"}


def make_workload(name, n, outdir):
    from carmel_b200 import synth
    if name == "cipher":
        return synth.write_cipher(outdir, n_lines=n, line_len=50)
    if name == "hmm":
        return synth.write_hmm(outdir, n_sent=n)
    raise SystemExit(f"unknown workload {name}")


def ensure_oracle():
    if not os.path.exists(ORACLE):
        subprocess.run(["make", "-C", os.path.join(ROOT, "oracle")], check=True, capture_output=True)


def cpu_oracle_throughput(w, sample_pairs, procs, budget_s=20.0):
    """arcs/s of the CPU oracle on the first `sample_pairs` examples, split over `procs` independent
    single-threaded processes (the reference is single threaded; examples are independent)."""
    ensure_oracle()
    d = tempfile.mkdtemp(prefix="cb200_cpu_")
    try:
        per = max(1, sample_pairs // procs)
        shards = []
        with open(w["files"][0]) as f:
            for i in range(procs):
                path = os.path.join(d, f"s{i}.data")
                k = 0
                with open(path, "w") as g:
                    while k < per:
                        a, b = f.readline(), f.readline()
                        if not b:
                            break
                        g.write(a)
                        g.write(b)
                        k += 1
                if k:
                    shards.append(path)
        t0 = time.time()  # calibrate the iteration count on shard 0 so the whole run stays near the budget
        r = subprocess.run([ORACLE, "--train-cascade", "-:", "--time-estimate=1", shards[0], *w["files"][1:]],
                           capture_output=True, text=True)
        j = json.loads(r.stdout.strip().splitlines()[-1])
        iters = int(max(1, min(50, budget_s / max(j["seconds"], 1e-3) / 2)))
        ps = [subprocess.Popen([ORACLE, "--train-cascade", "-:", f"--time-estimate={iters}", s, *w["files"][1:]],
                               stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True) for s in shards]
        outs = [json.loads(p.communicate()[0].strip().splitlines()[-1]) for p in ps]
        arcs = sum(o["trellis_arcs"] for o in outs)
        secs = max(o["seconds"] for o in outs)
        return {"value": arcs * iters / secs, "unit": UNIT, "cores": len(shards), "kind": "port",
                "sample": f"first {per * len(shards)} examples ({arcs} lattice arcs), {iters} cached EM iterations "
                          f"(-: semantics), {len(shards)} independent single-threaded oracle processes; "
                          f"calibration {time.time() - t0:.1f}s"}
    finally:
        shutil.rmtree(d, ignore_errors=True)


def oracle_example_lnp(w, n_pairs):
    """per-example ln P of the first n_pairs examples at the initial (normalised) weights, from the CPU oracle"""
    import numpy as np
    from carmel_b200 import synth
    ensure_oracle()
    d = tempfile.mkdtemp(prefix="cb200_par_")
    try:
        n = synth.head_corpus(w["files"][0], os.path.join(d, "s.data"), n_pairs)
        subprocess.run([ORACLE, "--train-cascade", f"--dump-estimate={d}/est", os.path.join(d, "s.data"), *w["files"][1:]],
                       capture_output=True, text=True, check=True)
        raw = open(f"{d}/est", "rb").read()
        n_arcs, n_ex = np.frombuffer(raw[:8], np.uint32)
        lnp = np.frombuffer(raw[8 + 16 * int(n_arcs):], np.float64, count=int(n_ex))
        assert int(n_ex) == n, (n_ex, n)
        return lnp.copy()
    finally:
        shutil.rmtree(d, ignore_errors=True)


def dump_outputs(outdir, arrays, limit=DUMP_BYTES):
    """write every array as outdir/<name>.npy in float64; when together they exceed `limit` bytes, arrays above 1 MB
    share what the smaller ones leave, each the same share of its elements, chosen by a fixed seed so that two runs
    keep the same indices"""
    import numpy as np
    os.makedirs(outdir, exist_ok=True)
    arrays = {k: np.ascontiguousarray(v, dtype=np.float64).ravel() for k, v in arrays.items()}
    small = sum(v.nbytes for v in arrays.values() if v.nbytes <= 1 << 20)
    large = sum(v.nbytes for v in arrays.values()) - small
    for name, v in arrays.items():
        if small + large > limit and v.nbytes > 1 << 20:
            keep = v.size * (limit - small) // large
            v = v[np.sort(np.random.default_rng(0).choice(v.size, keep, replace=False))]
        np.save(os.path.join(outdir, f"{name}.npy"), v)


def measure_tf32_peak(torch):
    """dense TF32 GEMM rate of this GPU (torch.matmul, 8192^3, best of 5): the denominator of the dense-state roofline"""
    old = torch.backends.cuda.matmul.allow_tf32
    try:
        torch.backends.cuda.matmul.allow_tf32 = True
        n = 8192
        a = torch.randn(n, n, device="cuda")
        b = torch.randn(n, n, device="cuda")
        best = 0.0
        for _ in range(2):
            a @ b
        for _ in range(5):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            a @ b
            e1.record()
            torch.cuda.synchronize()
            best = max(best, 2.0 * n ** 3 / (e0.elapsed_time(e1) / 1e3) / 1e12)
        return best
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default="cipher", choices=["cipher", "hmm", "forest", "gibbs"],
                    help="cipher (default): the full line with all legs; hmm / forest / gibbs: that workload's line alone")
    ap.add_argument("--precision", type=int, default=None, choices=[32, 64],
                    help="score precision (default 64 for cipher/hmm like carmel, 32 for forest like forest-em)")
    ap.add_argument("--space", default="scaled", choices=["scaled", "log"])
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--scale", type=int, default=1, help="corpus multiplier")
    ap.add_argument("--keep", action="store_true")
    ap.add_argument("--no-dense", action="store_true", help="single-workload runs: force the lattice (sparse) path")
    ap.add_argument("--no-sparse-leg", action="store_true", help="single-workload runs: skip the other path's measurement")
    ap.add_argument("--legs", default="all", help="all | none | comma list of c2,c3,c5,c4,cli")
    ap.add_argument("--c3-sentences", type=int, default=C3_SENTENCES)
    ap.add_argument("--unlock-lm", action="store_true",
                    help="cipher: make the bigram LM trainable too (transition counts are then part of the E-step)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the main line's last timed EM iteration computed as DIR/<name>.npy (see the module doc)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and (a.impl == "reference" or a.workload in ("forest", "gibbs")):
        ap.error("--dump-outputs writes the outputs of the B200 EM path (--workload cipher or hmm)")
    a.warmup = max(3, a.warmup)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if a.precision is None:
        a.precision = 32 if a.workload == "forest" else 64
    if a.workload == "forest":  # forest-em inside-outside (configs[4]) alone: see bench_forest.py
        import bench_forest
        if a.impl == "reference":
            if rank == 0:
                bench_forest.reference_arm(a)
            return
        bench_forest.run(a, rank, world, local)
        return
    if a.workload == "gibbs":  # --crp Gibbs sampling (configs[3]) alone: see bench_gibbs.py
        import bench_gibbs
        if a.impl == "reference":
            if rank == 0:
                bench_gibbs.reference_arm(a)
            return
        bench_gibbs.run(a, rank, world, local)
        return
    single = a.workload == "hmm" or a.no_dense or a.no_sparse_leg or a.scale != 1 or a.unlock_lm  # a development run
    legs = set() if (single or a.legs == "none") else ({"c2", "c3", "c5", "c4", "cli"} if a.legs == "all" else set(a.legs.split(",")))
    config = main_config(world)
    if single:
        config["workload"] = {"cipher": f"cipher ({CIPHER_LINES * a.scale} lines x 50 per GPU, development run)",
                              "hmm": f"configs[2] HMM tagging-style FST: 32 tags, 5k vocab, 4 tags/word, {125000 * a.scale} "
                                     "sentences per GPU (development run)"}[a.workload]

    # ---------------------------------------------------------------- reference arm (CPU oracle)
    if a.impl == "reference":
        if rank != 0:
            return
        d = tempfile.mkdtemp(prefix="cb200_ref_")
        try:
            w = make_workload(a.workload, CIPHER_LINES if a.workload == "cipher" else 125000, d)
            procs = max(1, os.cpu_count() or 1)
            n_pairs = CIPHER_SAMPLE if a.workload == "cipher" else C3_SAMPLE
            t0 = time.time()
            cb = cpu_oracle_throughput(w, n_pairs, procs, budget_s=8.0 * max(1, min(a.steps, 4)))
            line = {"metric": METRIC, "value": cb["value"], "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
                    "warmup": a.warmup, "ms_per_step": None, "higher_is_better": True, "scaling": "weak",
                    "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config, "impl": "reference",
                    "cpu_baseline": cb,
                    "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                    "note": "the reference binary needs Boost (absent, no network): this arm times the CPU oracle, a "
                            "restatement of the reference algorithm with the same class of data structures, on a bounded "
                            "sample of the same corpus (each step = one cached EM iteration over the sample)",
                    "wall_s": time.time() - t0}
            print(json.dumps(line))
        finally:
            shutil.rmtree(d, ignore_errors=True)
        return

    # ---------------------------------------------------------------- B200 arm
    import numpy as np
    import torch
    import torch.distributed as dist
    import carmel_b200 as cb

    assert torch.cuda.is_available(), "bench.py needs a GPU (carmel_b200 has no CPU fallback)"
    torch.cuda.set_device(local)
    gloo = None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        gloo = dist.new_group(backend="gloo")  # CPU side channel: survives a broken CUDA context on some rank (run_leg)
    shared = os.path.join(tempfile.gettempdir(), f"cb200_bench_{os.environ.get('MASTER_PORT', 'single')}_{os.getppid() if world > 1 else os.getpid()}")
    if rank == 0:
        shutil.rmtree(shared, ignore_errors=True)
        os.makedirs(shared, exist_ok=True)

    def barrier():
        if world > 1:
            dist.barrier()

    def trace(msg):  # CB200_BENCH_TRACE=1: where is every rank (multi-GPU debugging)
        if os.environ.get("CB200_BENCH_TRACE"):
            print(f"[bench rank {rank} +{time.time() - T0:.1f}s] {msg}", file=sys.stderr, flush=True)

    T0 = time.time()

    def new_token():
        """NCCL rendezvous token for one job's communicator (rank 0 makes it, everybody gets it)"""
        if world == 1:
            return None
        box = [cb.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        return box[0]

    def shared_workload(name, n, sub):
        """rank 0 writes the corpus + model files once; every rank reads the description"""
        d = os.path.join(shared, sub)
        if rank == 0:
            w = make_workload(name, n, d)
            if a.unlock_lm and name == "cipher":
                lm = w["files"][1]
                open(lm, "w").write(open(lm).read().replace("!))", "))"))
            json.dump(w, open(os.path.join(d, "workload.json"), "w"))
        barrier()
        return json.load(open(os.path.join(d, "workload.json")))

    stream = torch.cuda.Stream()
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")  # > 126 MB L2
    peaks, which = measured_peaks()
    hbm_peak = float(peaks.get("hbm_gbs", FALLBACK_HBM_GBS))
    tf32 = {"value": None}

    def measure(w, no_dense: bool, precision: int, steps: int, sample_pairs: int, shard: bool, traffic_key=None,
                check_n: bool = False, dump_dir=None) -> dict:
        """one job on workload w: warm-up + timed steps + e2e loop + kernel-alone pass + parity; returns what rank 0 prints.
        dump_dir: rank 0 writes the outputs of the last timed step there (dump_outputs)"""
        extra = ["-q", f"--gpu={local}"]
        if precision == 32:
            extra.append("--float")
        if a.space == "scaled":
            extra.append("--scaled")
        if no_dense:
            extra.append("--no-dense")
        if world > 1 and shard:
            extra.append(f"--shard={rank}/{world}")
        t_build = time.time()
        trace(f"measure: open job {extra}")
        job = cb.Job(extra + list(w["argv"]), comm_token=new_token() if (world > 1 and shard) else None)
        trace("prepare")
        ctx = job.prepare()
        ctx.set_stream(stream.cuda_stream)
        t_build = time.time() - t_build
        trace(f"prepared in {t_build:.1f}s")
        info = job.stats()
        dense = ctx.dense_stats()
        is_dense = dense["sequences"] > 0
        arcs_local, states_local = info["trellis_arcs"], info["trellis_states"]
        tot = torch.tensor([arcs_local, states_local, info["examples"], dense["positions"]], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(tot)
        arcs_total, states_total, ex_total, pos_total = (float(x) for x in tot.tolist())
        rs = precision // 8
        tol = 1e-6 if precision == 64 else 1e-4

        # ---- parity: per-example ln P at the initial weights against the CPU oracle (rank 0's block starts at example 0)
        parity = None
        if rank == 0 and sample_pairs:
            try:
                n = int(min(sample_pairs, info["examples"]))
                want = oracle_example_lnp(w, n)
                ctx.estimate()
                got = ctx.example_logprob(n)
                rel = float(np.max(np.abs(got - want) / np.maximum(1.0, np.abs(want))))
                parity = {"n": n, "max_rel": rel, "tol": tol, "ok": bool(rel <= tol),
                          "what": "per-example ln P at the initial weights, GPU path vs CPU oracle, first n examples"}
            except Exception as ex:
                parity = {"n": 0, "max_rel": None, "ok": False, "error": str(ex)[:300]}
        barrier()
        trace("first em_step")
        first = ctx.em_step(1.0)  # (first call: plain pass + graph capture)
        trace("first em_step done")
        first_counts = ctx.counts() if check_n and rank == 0 else None
        # the dense-state path's working set (symbols + alpha rows) fits in L2: flush L2 between its timed steps
        flush = is_dense

        def timed(fn, n_steps):
            barrier()
            torch.cuda.synchronize()
            total = 0.0
            if not flush:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                with torch.cuda.stream(stream):
                    e0.record()
                    for _ in range(n_steps):
                        fn()
                    e1.record()
                torch.cuda.synchronize()
                total = e0.elapsed_time(e1)
            else:
                for _ in range(n_steps):
                    with torch.cuda.stream(stream):
                        flush_buf.fill_(1)
                        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        e0.record()
                        fn()
                        e1.record()
                    torch.cuda.synchronize()
                    total += e0.elapsed_time(e1)
            barrier()
            ms = torch.tensor([total], dtype=torch.float64, device="cuda")
            if world > 1:
                dist.all_reduce(ms, op=dist.ReduceOp.MAX)
            return float(ms.item())

        last = [first]

        def step():
            last[0] = ctx.em_step(1.0)

        for _ in range(a.warmup):
            step()
        sampler = ClockSampler(local)
        if rank == 0:
            sampler.start()
        l0, c0 = ctx.launch_count(), ctx.collective_count()
        trace("timed region")
        ms = timed(step, steps)
        trace("timed region done")
        launches, collectives = ctx.launch_count() - l0, ctx.collective_count() - c0
        clocks = sampler.stop() if rank == 0 else None
        value = arcs_total * steps / (ms / 1e3)
        if dump_dir and rank == 0:  # before the e2e loop below runs further EM iterations
            r_last, change = last[0]
            dump_outputs(dump_dir, {"step_result": [r_last.sum_ln_p, r_last.sum_w_ln_p, r_last.n_zero, change],
                                    "params": ctx.get_params(), "counts": ctx.counts(),
                                    "example_ln_p": ctx.example_logprob(int(info["examples"]))})

        # ---- e2e: host buffers through the C ABI every step
        n_params, n_arcs = info["n_params"], info["n_arcs"]
        h_params = torch.empty(n_params, dtype=torch.float64).pin_memory()
        n_slots = ctx.count_slots()
        h_counts = torch.empty(n_slots, dtype=torch.float64).pin_memory()
        ctx.get_params_ptr(h_params.data_ptr())

        def e2e_step():
            ctx.set_params_ptr(h_params.data_ptr())           # H2D: parameter vector
            ctx.em_step(1.0)                                  # E-step, all-reduce, M-step; D2H: likelihood + max change
            ctx.get_counts_ptr(h_counts.data_ptr(), n_slots)  # D2H: expected counts (one per count slot)
            ctx.get_params_ptr(h_params.data_ptr())           # D2H: new parameters

        for _ in range(2):
            e2e_step()
        ms_e2e = timed(e2e_step, steps)
        e2e = {"value": arcs_total * steps / (ms_e2e / 1e3), "unit": UNIT, "h2d_bytes_per_step": 8 * n_params,
               "d2h_bytes_per_step": 8 * n_params + 8 * n_slots + 32, "ms_per_step": ms_e2e / steps,
               "lattices": ("never materialised (dense-state view): symbol sequences resident; one-time host prep + upload "
                            if is_dense else "resident (carmel -: derivation-cache semantics); one-time host build + "
                            "flatten + upload ") + f"took {t_build:.2f}s on this rank"}

        # ---- the E-step kernel alone: CUDA events around it (un-graphed pass: events cannot be read out of a graph)
        fb = []
        for _ in range(max(3, min(steps, 10))):
            if flush:
                with torch.cuda.stream(stream):
                    flush_buf.fill_(1)
            ctx.estimate_launch()
            ctx.allreduce_counts()
            ctx.estimate_finish()
            fb.append(ctx.last_fb_time_ms())
        k_ms = sum(m for m, _ in fb) / len(fb)
        n_k = fb[0][1]

        res = {"is_dense": is_dense, "value": value, "ms": ms, "steps": steps, "e2e": e2e, "launches": int(launches),
               "collectives": int(collectives), "clocks": clocks, "parity": parity, "first": first,
               "totals": {"examples": ex_total, "trellis_arcs": arcs_total, "trellis_states": states_total,
                          "n_params": n_params, "n_arcs": n_arcs}, "count_slots": n_slots, "l2_flush": flush}
        if rank == 0:
            if is_dense and dense["kernel"] == "sparse":
                # sparse-emission kernel: per position one symbol, K alpha values written + read, one exponent written +
                # read; emission rows / transition matrix come from L2 / shared memory
                res["totals"]["positions"] = pos_total
                K = dense["k"]
                bytes_pos = 2.0 + 2.0 * K * rs + 8.0
                ach = bytes_pos * dense["positions"] / (k_ms / 1e3) / 1e9
                lattice_bytes = (16.0 + 2.0 * rs * (states_local / max(1, arcs_local))) * arcs_local
                res["roofline"] = {
                    "bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak,
                    "traffic": measured_traffic("k_fb_sparse", dense["positions"]) if traffic_key else None, "peak_source": which,
                    "kernel": "k_fb_sparse (forward + backward + counts, one sequence per lane, lattices never "
                              "materialised; 1 launch per iteration)",
                    "kernel_ms": k_ms, "algorithmic_bytes_per_position": bytes_pos,
                    "positions_per_launch": dense["positions"], "kernel_share_of_step": k_ms / (ms / steps),
                    "lattice_equivalent": {
                        "note": "what the same arcs would cost as streamed lattice records (SURVEY 8d: 16 B/arc + alpha): "
                                "this kernel does not read them, so this is NOT a roofline fraction",
                        "algorithmic_bytes": lattice_bytes, "achieved_gbs": lattice_bytes / (k_ms / 1e3) / 1e9}}
                res["layout"] = dense
            elif is_dense:
                res["totals"]["positions"] = pos_total
                S = dense["n_states"]  # useful flops (SURVEY 8d: S x S mat-vecs); the kernel computes on 32 padded lanes
                products = 3 if dense["t_slots"] else 2  # alpha, beta (+ xi when transitions are trainable)
                flops = 2.0 * products * S * S * dense["positions"]
                if tf32["value"] is None:
                    tf32["value"] = measure_tf32_peak(torch)
                ach = flops / (k_ms / 1e3) / 1e12
                hbm_bytes = dense["positions"] * (2.0 * 32 * rs + 8 + 2 + 2)  # alpha row written + read, exponents, symbol twice
                res["roofline"] = {
                    "bound": "tensor", "achieved": ach, "peak": tf32["value"], "unit": "TFLOP/s", "frac": ach / tf32["value"],
                    "traffic": measured_traffic("k_fb_dense", dense["positions"]) if traffic_key else None,
                    "peak_source": "TF32 GEMM rate measured in this run (torch.matmul 8192^3, allow_tf32, best of 5)",
                    "kernel": ("k_dense_tc<fwd> + k_dense_tc<bwd> + k_dense_tc_counts (3xTF32 mma.sync sweeps, 16 sequences per "
                               "warp; 3 launches per iteration)" if dense["kernel"] == "dense_tc" else
                               "k_fb_dense (forward + backward + counts over never-materialised lattices, 1 launch per iteration)"),
                    "kernel_ms": k_ms, "flops_per_position": 2.0 * products * S * S, "positions_per_launch": dense["positions"],
                    "kernel_share_of_step": k_ms / (ms / steps),
                    "note": ("tensor-core path: each position step of 16 sequences is a [16x32].[32x32] product in 3xTF32"
                             if dense["kernel"] == "dense_tc" else
                             "CUDA-core FMA kernel (fp32/fp64), one warp per sequence: a serial chain of line_len dependent 32x32 "
                             "mat-vecs, latency bound at this corpus size (0.3 GFLOP per iteration); reported against the tensor "
                             "peak as SURVEY 8(d) asks for the dense case"),
                    "hbm_equivalent": {"algorithmic_bytes": hbm_bytes, "achieved_gbs": hbm_bytes / (k_ms / 1e3) / 1e9,
                                       "peak_gbs": hbm_peak}}
                res["layout"] = dense
            else:
                bytes_per_arc = 16.0 + 2.0 * rs * (states_local / max(1, arcs_local))
                achieved = bytes_per_arc * arcs_local / (k_ms / 1e3) / 1e9
                lay = {**ctx.layout_stats(), **ctx.lane_stats(), **ctx.wide_stats()}
                kname = ("k_fb_wide (warp per lattice, bulk-copy record stream, factored weights in shared memory)"
                         if lay["wide_examples"] else "k_fb_lane (lattice per lane, tiles of 32)" if lay["lane_examples"] else "k_fb_ell / k_fb_warp")
                traffic = measured_traffic(traffic_key, arcs_local) if traffic_key else None
                res["roofline"] = {"bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s",
                                   "frac": achieved / hbm_peak, "traffic": traffic,
                                   "traffic_over_algorithmic": (traffic / (bytes_per_arc * arcs_local)) if traffic else None,
                                   "peak_source": which, "kernel": f"{kname}: forward + backward + counts, {n_k} launch(es) per iteration",
                                   "kernel_ms": k_ms, "algorithmic_bytes_per_arc": bytes_per_arc,
                                   "arcs_per_launch_set": arcs_local, "kernel_share_of_step": k_ms / (ms / steps),
                                   "timing": "CUDA events around the kernel on the launching stream, un-graphed pass after the "
                                             "timed region (the timed region replays a CUDA graph)"}
                res["layout"] = lay
        trace("close job")
        job.close()
        trace("job closed")

        # ---- N > 1: the same total corpus on rank 0 alone; sum ln P and the reduced count table must agree
        if check_n and world > 1:
            if rank == 0:
                try:
                    job1 = cb.Job(extra[:-1] + list(w["argv"]))  # (without --shard)
                    ctx1 = job1.prepare()
                    r1, _ = ctx1.em_step(1.0)
                    c1 = ctx1.counts()
                    job1.close()
                    r0 = first[0]
                    rel_p = abs(r0.sum_ln_p - r1.sum_ln_p) / max(1.0, abs(r1.sum_ln_p))
                    rel_c = float(np.max(np.abs(first_counts - c1) / np.maximum(1e-300, np.maximum(np.abs(c1), 1e-12))))
                    res["parity_n"] = {"ranks": world, "sum_ln_p_sharded": r0.sum_ln_p, "sum_ln_p_one_rank": r1.sum_ln_p,
                                       "rel_sum_ln_p": rel_p, "max_rel_counts": rel_c, "tol": 1e-9,
                                       "ok": bool(rel_p <= 1e-9 and rel_c <= 1e-9 and r0.n_zero == r1.n_zero),
                                       "what": "first EM iteration: N-rank sharded E-step + NCCL all-reduce vs rank 0 alone over "
                                               "the same total corpus, through the same kernels"}
                except Exception as ex:
                    res["parity_n"] = {"ranks": world, "ok": False, "error": str(ex)[:300]}
            barrier()
        return res

    def leg_of(res, note):
        return {"value": res["value"], "unit": UNIT, "ms_per_step": res["ms"] / res["steps"], "steps": res["steps"],
                "roofline": res.get("roofline"), "e2e": res["e2e"], "parity": res["parity"], "layout": res.get("layout"),
                "totals": res["totals"], "count_slots": res["count_slots"], "gpu_launches": res["launches"],
                "collectives": res["collectives"], "l2_flush": res["l2_flush"], "note": note,
                **({"parity_n": res["parity_n"]} if "parity_n" in res else {})}

    # ---------------------------------------------------------------- main line
    if single:
        w = shared_workload(a.workload, (CIPHER_LINES if a.workload == "cipher" else 125000) * a.scale * world, "main")
        main_res = measure(w, a.no_dense, a.precision, a.steps, CIPHER_SAMPLE if a.workload == "cipher" else C3_SAMPLE, True,
                           traffic_key=None, dump_dir=a.dump_outputs)
        other = None
        if main_res["is_dense"] and not a.no_sparse_leg:
            other = measure(w, True, a.precision, a.steps, 0, True)
    else:
        w = shared_workload("cipher", CIPHER_LINES * world, "main")
        main_res = measure(w, True, 64, a.steps, CIPHER_SAMPLE, True, traffic_key="k_fb_wide_cipher", check_n=True,
                           dump_dir=a.dump_outputs)
    line = None
    if rank == 0:
        failures = []
        line = {"metric": METRIC, "value": main_res["value"], "unit": UNIT, "n_gpus": world, "steps": a.steps,
                "warmup": a.warmup, "ms_per_step": main_res["ms"] / a.steps, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f64" if a.precision == 64 else "f32", "data": "synthetic", "config": config,
                "path": ("lattice path (--no-dense): derivation lattices materialised, resident and streamed every iteration -- "
                         "the sparse-trellis forward/backward the HBM-roofline target is quoted on; the product's default for "
                         "this model is the dense-state path, reported in dense_path") if not single else
                        ("dense-state" if main_res["is_dense"] else "lattice"),
                "roofline": main_res.get("roofline"), "parity": main_res["parity"], "e2e": main_res["e2e"],
                "gpu_launches": main_res["launches"], "collectives": main_res["collectives"], "clocks": main_res["clocks"],
                "totals": main_res["totals"], "layout": main_res.get("layout"), "count_slots": main_res["count_slots"]}
        if "parity_n" in main_res:
            line["parity_n"] = main_res["parity_n"]
        if single and other is not None:
            line["sparse_path"] = leg_of(other, "same corpus with --no-dense")

    def finish_line():
        """rank 0: parity gates, then THE line"""
        if tf32["value"] is not None:
            line["tf32_peak_tflops_measured"] = tf32["value"]
        # parity gates: a line whose GPU results differ from the oracle's is not a measurement
        bad = []
        for key in ("parity", "parity_n"):
            if key in line and line[key] is not None and not line[key].get("ok", False):
                bad.append(key)
        for leg in ("dense_path", "c3", "c5", "c4"):
            p = (line.get(leg) or {}).get("parity")
            if p is not None and not p.get("ok", False):
                bad.append(f"{leg}.parity")
        line["parity_ok"] = not bad
        if bad:  # a line whose results differ from the oracle's is not a measurement: say so in the line itself
            line["parity_failures"] = bad
            line["invalid"] = "parity check failed: " + ", ".join(bad)
        print(json.dumps(line, default=lambda o: str(o)))

    # ---------------------------------------------------------------- legs
    def run_leg(name, fn):
        """a leg never takes the line down: failures are recorded in its place"""
        t0 = time.time()
        try:
            out = fn()
            if rank == 0 and out is not None:
                out["wall_s"] = time.time() - t0
                line[name] = out
        except Exception as ex:  # noqa: BLE001
            if rank == 0:
                line[name] = {"failed": f"{type(ex).__name__}: {ex}"[:400], "wall_s": time.time() - t0}
        # a CUDA error is sticky: if the device of ANY rank is broken after this leg, nothing later can run (and the
        # NCCL barrier would hang the other ranks) -- every rank learns it over the CPU group, rank 0 prints the line
        # with what it has, and all ranks leave
        broken = 0
        try:
            torch.cuda.synchronize()
        except Exception:  # noqa: BLE001
            broken = 1
        if gloo is not None:
            flag = torch.tensor([broken], dtype=torch.int32)
            dist.all_reduce(flag, op=dist.ReduceOp.MAX, group=gloo)
            broken = int(flag.item())
        if broken:
            if rank == 0:
                line["aborted_after_leg"] = name
                finish_line()
            sys.stdout.flush()
            os._exit(0)
        barrier()

    if "c2" in legs:
        def c2():
            flush_buf.fill_(0)
            r = measure(w, False, 64, a.steps, CIPHER_SAMPLE, True, traffic_key="k_fb_dense")
            return leg_of(r, "same corpus on the product's default path for this model: dense-state view, lattices never "
                             "materialised (k_fb_dense); weak scaling") if rank == 0 else None
        run_leg("dense_path", c2)

    if "c3" in legs:
        def c3():
            n_sent = a.c3_sentences
            w3 = shared_workload("hmm", n_sent, "c3")
            steps3 = max(3, min(a.steps, 5))
            rs_ = measure(w3, True, 64, steps3, C3_SAMPLE, True, traffic_key="k_fb_lane", check_n=False)
            rd_ = measure(w3, False, 64, steps3, 0, True, traffic_key="k_fb_sparse")
            if rank != 0:
                return None
            out = leg_of(rs_, "lattice path (--no-dense, k_fb_lane); count accumulation is bound by the fp64 RED rate of the "
                              "L2 atomic units (profiles/micro/red_bench.cu: 195 G updates/s on this GPU; 1.26 updates per arc)")
            out["config"] = {"workload": f"configs[2] HMM tagging-style FST: 32 tags, 5k vocab, 4 tags/word, {n_sent} sentences "
                                         f"IN TOTAL, sharded over {world} GPU(s)", "scaling": "strong"}
            out["scaling"] = "strong"
            out["dense_path"] = leg_of(rd_, "same corpus on the product's default path for this model (k_fb_sparse)")
            return out
        run_leg("c3", c3)

    if "c5" in legs:
        def c5():
            import bench_forest
            fa = argparse.Namespace(**vars(a))
            fa.precision, fa.scale = 32, 1
            fa.steps = max(3, min(a.steps, 10))
            return bench_forest.run(fa, rank, world, local, as_leg=True, token=new_token(), with_cpu=(world == 1))
        run_leg("c5", c5)

    if "c4" in legs:
        def c4():
            import bench_gibbs
            ga = argparse.Namespace(**vars(a))
            ga.scale = 4  # 20,000 lines x 50 = configs[3]'s 1M letters (in total: sharded over the ranks)
            ga.steps = max(3, min(a.steps, 10))
            ga.no_dense = False
            return bench_gibbs.run(ga, rank, world, local, as_leg=True, with_cpu=(world == 1), token=new_token())
        run_leg("c4", c4)

    if "cli" in legs and world == 1:
        def cli():
            # what a user of the drop-in sees: read + compose + lattice build + upload + 20 EM iterations + write
            from carmel_b200 import CLI_PATH, synth
            ensure_oracle()
            d = os.path.join(shared, "cli")
            os.makedirs(d, exist_ok=True)
            files = [shutil.copy(f, d) for f in w["files"]]
            out = {}
            for name, extra in (("lattice_path", ["--no-dense"]), ("default_path", [])):
                t0 = time.time()
                r = subprocess.run([CLI_PATH, "--train-cascade", "--scaled", "-M", "20", *extra, f"--history={d}/h.{name}", *files],
                                   capture_output=True, text=True, cwd=d)
                wall = time.time() - t0
                its = sum(1 for _ in open(f"{d}/h.{name}")) if os.path.exists(f"{d}/h.{name}") else 0
                out[name] = {"wall_s": wall, "iterations": its, "rc": r.returncode,
                             "arcs_per_s": main_res["totals"]["trellis_arcs"] * its / wall if wall > 0 else None}
            n = CIPHER_SAMPLE
            synth.head_corpus(files[0], os.path.join(d, "sample.data"), n)
            t0 = time.time()
            r = subprocess.run([ORACLE, "--train-cascade", "-M", "20", f"--history={d}/h.oracle", os.path.join(d, "sample.data"), *files[1:]],
                               capture_output=True, text=True, cwd=d)
            wall = time.time() - t0
            its = sum(1 for _ in open(f"{d}/h.oracle")) if os.path.exists(f"{d}/h.oracle") else 0
            arcs_sample = main_res["totals"]["trellis_arcs"] * n / max(1.0, main_res["totals"]["examples"])
            out["cpu_oracle_cli"] = {"wall_s": wall, "iterations": its, "rc": r.returncode, "examples": n, "cores": 1,
                                     "arcs_per_s": arcs_sample * its / wall if wall > 0 else None,
                                     "note": f"same command on the first {n} lines (one thread, lattices rebuilt every iteration "
                                             "like carmel without -:)"}
            out["what"] = "wall time of `carmel-b200 --train-cascade --scaled -M 20 cipher.data lm.wfsa channel.fst` (whole process)"
            return out
        run_leg("e2e_cli", cli)

    if rank == 0:
        try:
            cpu = cpu_oracle_throughput(w, CIPHER_SAMPLE if a.workload == "cipher" else C3_SAMPLE, max(1, os.cpu_count() or 1),
                                        budget_s=12.0) if world == 1 else None
        except Exception as ex:  # the bench line must still be printed
            cpu = {"value": None, "unit": UNIT, "cores": 0, "kind": "port", "sample": f"failed: {ex}"}
        if cpu is not None:
            line["cpu_baseline"] = cpu
        finish_line()
    barrier()
    if rank == 0 and not a.keep:
        shutil.rmtree(shared, ignore_errors=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
