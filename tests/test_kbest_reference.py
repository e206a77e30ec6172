"""The CPU reference for k-best lists (kbest_helpers.Lattices.kbest: a lazy enumeration with per-state candidate heaps
over the oracle's lattices, the restatement behind the --viterbi -k parity tests) against brute-force enumeration of
EVERY derivation of the dumped lattices, and the -k argument handling of the command line.  CPU only."""
import math
import os

import numpy as np
import pytest

from helpers import random_wfst, read_estimate_dump, read_trellis_dump, run, sample_pairs, stage
from kbest_helpers import Lattices, compare_kbest


def _random_case(tmp_path, seed):
    rng = np.random.default_rng(20271001 + seed)
    ns = int(rng.integers(2, 6))
    fst, ins, outs, arcs = random_wfst(rng, n_states=ns, eps_rate=float(rng.uniform(0, 0.3)))
    corpus = sample_pairs(rng, arcs, ns, n_pairs=8, max_steps=6, ins=ins, outs=outs)
    f, c = os.path.join(str(tmp_path), "r.fst"), os.path.join(str(tmp_path), "r.data")
    open(f, "w").write(fst)
    open(c, "w").write(corpus)
    return c, f


@pytest.mark.parametrize("seed", range(8))
def test_reference_kbest_is_the_top_k_of_all_derivations(oracle_bin, tmp_path, seed):
    c, f = _random_case(tmp_path, seed)
    d = str(tmp_path)
    rc, _, err = run(oracle_bin, ["-t", f"--dump-trellis={d}/t", f"--dump-estimate={d}/e", c, f])
    assert rc == 0, err
    rc, _, err = run(oracle_bin, ["-t", f"--dump-viterbi={d}/v", c, f])
    assert rc == 0, err
    lat = Lattices(read_trellis_dump(f"{d}/t"), read_estimate_dump(f"{d}/e")["ln_w"])
    n_ex = lat.t["n_ex"]
    assert n_ex >= 4
    every = [sorted(lat.paths(e), key=lambda x: -x[0]) for e in range(n_ex)]
    every = [[(w, p) for w, p in ps if w > -math.inf] for ps in every]
    most = max(len(ps) for ps in every)
    for k in (1, 3, 17, most + 2):
        for e in range(n_ex):
            got = lat.kbest(e, k)
            assert len(got) == k
            want = (every[e] + [(-math.inf, ())] * k)[:k]
            for r, ((ww, _), (gw, gp)) in enumerate(zip(want, got)):
                if ww == -math.inf:
                    assert gw == -math.inf and gp == (), (e, r, gw, gp)  # padding
                else:
                    assert abs(ww - gw) <= 1e-12 * max(1.0, abs(ww)), (e, r, ww, gw)
                    pw = lat.weight(e, gp)
                    assert pw is not None and abs(pw - gw) <= 1e-12 * max(1.0, abs(gw)), (e, r, gp, pw, gw)
            listed = [p for w, p in got if w > -math.inf]
            assert len(set(listed)) == len(listed), (e, listed)  # distinct paths
            compare_kbest(want, got, lambda p, e=e: lat.weight(e, p))
            if k == most + 2:
                assert got[-1][0] == -math.inf
    # rank 0 has the weight of the oracle's best-derivation pass
    best = [float(ln.split()[0]) for ln in open(f"{d}/v")]
    assert len(best) == n_ex
    for e in range(n_ex):
        w0 = lat.kbest(e, 1)[0][0]
        assert w0 == best[e] or abs(w0 - best[e]) <= 1e-12 * max(1.0, abs(w0)), (e, w0, best[e])


def test_k_argument(native_lib, tmp_path):
    """-k 0 / a non-number is refused with the argument-error exit code before any work; bundled value flags bind by
    carmel's priority chain, k before M: -Mk 0 3 is refused for k = 0, -Mk 3 0 is not"""
    from carmel_b200 import CLI_PATH
    c, f = _random_case(tmp_path, 0)
    d = str(tmp_path)
    for bad in ("0", "x", "-2", ""):
        rc, _, err = run(CLI_PATH, ["-t", f"--viterbi={d}/p", "-k", bad, c, f])
        assert rc == -9 % 256 and "-k needs" in err, (bad, rc, err)
        assert not os.path.exists(f"{d}/p")
    rc, _, err = run(CLI_PATH, ["-t", f"--viterbi={d}/p", "-Mk", "0", "3", c, f])
    assert rc == -9 % 256 and '-k needs a whole number of derivations >= 1 (got "0")' in err, (rc, err)
    rc, _, err = run(CLI_PATH, ["-t", f"--viterbi={d}/p", "-Mk", "3", "0", c, f])
    assert "-k needs" not in err, err
    # without --viterbi, -k is accepted and unused: no refusal
    rc, _, err = run(CLI_PATH, ["-t", "-M", "0", "-k", "0", c, f])
    assert "-k needs" not in err, err


def test_kbest_without_gpu_fails_loudly(native_lib, tmp_path):
    """--viterbi -k 5 on a machine without a CUDA device stops with the no-CPU-fallback error and writes nothing"""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    from carmel_b200 import CLI_PATH
    paths = stage(tmp_path, "cipher.data", "cipher.wfsa", "cipher.fst")
    rc, _, err = run(CLI_PATH, ["--train-cascade", f"--viterbi={tmp_path}/v", "-k", "5", *paths])
    assert rc != 0 and ("no CPU fallback" in err or "CUDA" in err), err
    assert not (tmp_path / "v").exists() or (tmp_path / "v").stat().st_size == 0


def test_gpus_refuses_viterbi(native_lib, tmp_path):
    """--viterbi decodes on one GPU: --gpus=2 --viterbi is refused instead of training"""
    from carmel_b200 import CLI_PATH
    paths = stage(tmp_path, "cipher.data", "cipher.wfsa", "cipher.fst")
    rc, _, err = run(CLI_PATH, ["--train-cascade", "--gpus=2", f"--viterbi={tmp_path}/v", "-k", "3", *paths])
    assert rc != 0 and "--viterbi decodes on one GPU" in err, err
    assert not (tmp_path / "v").exists()
