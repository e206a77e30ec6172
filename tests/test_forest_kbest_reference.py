"""The CPU reference for forest k-best lists (forest_kbest_helpers.ForestRef.kbest: a lazy enumeration with a candidate
heap per node over the library's pre-order arrays, the restatement behind the -v --kbest parity tests) against
brute-force enumeration of EVERY derivation (forest_helpers.enumerate_derivations), and the --kbest argument handling
of forest-em-b200.  CPU only."""
import math
import os
from collections import Counter

import numpy as np
import pytest

from forest_helpers import enumerate_derivations, parse_forest, random_forest, random_normgroups
from forest_kbest_helpers import ForestRef, compare_kbest, forests_to_arrays
from helpers import run


def _count(ref, v, memo):
    """number of derivations of real node v (zero weights included)"""
    if v not in memo:
        if ref.lb[v]:
            memo[v] = math.prod(_count(ref, c, memo) for c in ref.slots[v])
        else:
            memo[v] = sum(_count(ref, c, memo) for c in ref.slots[v])
    return memo[v]


@pytest.mark.parametrize("seed", range(6))
def test_reference_kbest_is_the_top_k_of_all_derivations(seed):
    rng = np.random.default_rng(20271101 + seed)
    n_rules = 12
    texts = []
    while len(texts) < 50:  # a few hundred over the seeds, small enough to enumerate
        t = random_forest(rng, n_rules, depth=int(rng.integers(1, 4)), share=0.25)
        no, nx, lb, br = forests_to_arrays([t])
        if _count(ForestRef(nx, lb, br, np.zeros(n_rules + 1)), 0, {}) <= 3000:
            texts.append(t)
    # weights with exact ties (repeated values) and zero-weight rules
    p = rng.choice([0.0, 0.25, 0.5, 0.5, 1.0, 0.125], size=n_rules + 1)
    with np.errstate(divide="ignore"):
        ln_w = np.log(p)
    for t in texts:
        no, nx, lb, br = forests_to_arrays([t])
        root, defs = parse_forest(t)
        every = [(math.log(q), c) for q, c in enumerate_derivations(root, defs, {r: p[r] for r in range(n_rules + 1)})
                 if q > 0]
        every.sort(key=lambda x: -x[0])
        for k in (1, 3, 17, len(every) + 2):
            ref = ForestRef(nx, lb, br, ln_w)
            got = ref.kbest(k)
            assert len(got) == k
            for r, (gw, gp) in enumerate(got):
                if r >= len(every):
                    assert gw == -math.inf and gp == ()
                    continue
                assert abs(gw - every[r][0]) <= 1e-12 * max(1.0, abs(gw)), (t, r, gw, every[r][0])
                sw = ref.score_of(gp)
                assert sw is not None and abs(sw - gw) <= 1e-12 * max(1.0, abs(gw)), (t, gp, sw, gw)
            if k >= len(every):  # the whole list: the same multiset of (rule uses) as the brute force
                key = lambda c: tuple(sorted(c.items()))
                want = sorted(key(c) for _, c in every)
                have = sorted(key(Counter(int(lb[x]) for x in gp)) for _, gp in got if gp)
                assert want == have, t
                compare_kbest(got, got, ref.score_of)


def test_reference_on_a_deep_chain():
    """200 nested AND / OR levels with a shared node at every level: the lazy reference and the rule's score walk"""
    body = "1"
    for d in range(200):
        body = f"(OR #{d + 1}(2 {body}) (3 #{d + 1}))"
    no, nx, lb, br = forests_to_arrays([body])
    ln_w = np.log(np.array([1.0, 0.5, 0.25, 0.75]))
    ref = ForestRef(nx, lb, br, ln_w)
    got = ref.kbest(5)
    assert all(w > -math.inf for w, _ in got)
    for w, s in got:
        assert abs(ref.score_of(s) - w) <= 1e-9 * abs(w)
    assert [w for w, _ in got] == sorted((w for w, _ in got), reverse=True)


@pytest.fixture(scope="module")
def fem(native_lib):
    from carmel_b200 import FOREST_CLI_PATH
    return FOREST_CLI_PATH


def test_kbest_argument(fem, tmp_path):
    """--kbest=n is refused with forest-em's argument-error exit (1, ERROR: ...) before any work: without -v, 0, a
    non-number, and with --shard / --gpus=N"""
    d = str(tmp_path)
    rng = np.random.default_rng(3)
    open(f"{d}/f", "w").write("\n".join(random_forest(rng, 10, depth=3) for _ in range(5)) + "\n")
    open(f"{d}/n", "w").write(random_normgroups(rng, 10))
    base = ["-f", f"{d}/f", "-n", f"{d}/n", "-i", "2"]
    for bad in ("0", "x", "-2", "", "3x"):
        rc, _, err = run(fem, [*base, "-v", f"{d}/v", f"--kbest={bad}"])
        assert rc == 1 and "ERROR: --kbest=n needs a whole number" in err, (bad, rc, err)
        assert not os.path.exists(f"{d}/v")
    rc, _, err = run(fem, [*base, "-v", f"{d}/v", "--kbest"])
    assert rc == 1 and "ERROR: --kbest=n needs a whole number" in err, err
    rc, _, err = run(fem, [*base, "--kbest=3"])
    assert rc == 1 and "ERROR: --kbest=n needs -v" in err, err
    rc, _, err = run(fem, [*base, "-v", f"{d}/v", "--kbest=3", "--shard=0/2"])
    assert rc == 1 and "ERROR: --kbest decodes on one GPU" in err, err
    rc, _, err = run(fem, [*base, "-v", f"{d}/v", "--kbest=3", "--gpus=2"])
    assert rc == 1 and "ERROR: --kbest decodes on one GPU" in err, err
    assert not os.path.exists(f"{d}/v")


def test_kbest_without_gpu_fails_loudly(fem, tmp_path):
    """-v --kbest=5 on a machine without a CUDA device stops with an error and writes no k-best file"""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    d = str(tmp_path)
    rng = np.random.default_rng(4)
    open(f"{d}/f", "w").write("\n".join(random_forest(rng, 10, depth=3) for _ in range(5)) + "\n")
    open(f"{d}/n", "w").write(random_normgroups(rng, 10))
    rc, _, err = run(fem, ["-f", f"{d}/f", "-n", f"{d}/n", "-i", "2", "-v", f"{d}/v", "--kbest=5"])
    assert rc != 0 and "ERROR" in err, err
    assert not os.path.exists(f"{d}/v") or os.path.getsize(f"{d}/v") == 0
