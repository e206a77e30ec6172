"""The CPU reference for forest sums and samples (forest_sample_helpers.ForestSampler: inside by memoised recursion over
the library's pre-order arrays, a recursive pre-order walk per sample, the restatement behind the -v --sample parity
tests) against brute-force enumeration (forest_helpers.brute_force), its draws against the enumerated probabilities,
and the --sample argument handling of forest-em-b200.  CPU only."""
import math
import os

import numpy as np
import pytest

from forest_helpers import brute_force, random_forest, random_normgroups
from forest_kbest_helpers import ForestRef, forests_to_arrays
from forest_sample_helpers import ForestSampler, chi2_fit, small_forests
from helpers import run


def _weights(rng, n_rules):
    """probabilities with exact ties (repeated values) and zero-weight rules, and their logs"""
    p = rng.choice([0.0, 0.25, 0.5, 0.5, 1.0, 0.125, 0.9], size=n_rules + 1)
    with np.errstate(divide="ignore"):
        return p, np.log(p)


@pytest.mark.parametrize("seed", range(4))
def test_reference_totals_are_the_enumerated_sums(seed):
    rng = np.random.default_rng(20281101 + seed)
    n_rules = 12
    p, ln_w = _weights(rng, n_rules)
    n_zero = 0
    for t in small_forests(rng, 40, n_rules, max_derivations=400):
        _, nx, lb, br = forests_to_arrays([t])
        s = ForestSampler(nx, lb, br, ln_w)
        want, _ = brute_force(t, {r: p[r] for r in range(n_rules + 1)})
        got = s.ln_total()
        if want == 0:
            n_zero += 1
            assert got == -math.inf, (t, got)
            assert s.draw(1, 0, 3)[0] == [()] * 3
            continue
        assert abs(got - math.log(want)) <= 1e-12 * max(1.0, abs(got)), (t, got, math.log(want))
        every = s.derivations()
        assert abs(math.log(sum(math.exp(w) for w in every.values())) - got) <= 1e-12 * max(1.0, abs(got))
    assert n_zero < 40


def test_reference_draws_follow_the_enumerated_probabilities():
    """12 forests with back references and zero-weight rules, 10,000 draws each at a fixed seed: chi-square fit"""
    rng = np.random.default_rng(20281201)
    n_rules = 10
    p, ln_w = _weights(rng, n_rules)
    fitted = 0
    for i, t in enumerate(small_forests(rng, 200, n_rules)):
        _, nx, lb, br = forests_to_arrays([t])
        s = ForestSampler(nx, lb, br, ln_w)
        if s.ln_total() == -math.inf or len(s.derivations()) < 2:
            continue
        paths, w, ex = s.draw(7, i, 10000)
        ref = ForestRef(nx, lb, br, ln_w)
        for q, x in zip(paths[:50], w[:50]):
            assert abs(ref.score_of(q) - x) <= 1e-12 * max(1.0, abs(x)), (q, x)
        assert chi2_fit(s, paths) > 1e-6, t
        fitted += 1
        if fitted == 12:
            break
    assert fitted == 12


def test_reference_walks_in_pre_order_and_deep():
    """the recorded nodes are the derivation's AND nodes in pre-order (the -v tree reads them back), 200 levels deep"""
    body = "1"
    for d in range(200):
        body = f"(OR #{d + 1}(2 {body}) (3 #{d + 1}))"
    _, nx, lb, br = forests_to_arrays([body])
    ln_w = np.log(np.array([1.0, 0.5, 0.25, 0.75]))
    s, ref = ForestSampler(nx, lb, br, ln_w), ForestRef(nx, lb, br, ln_w)
    paths, w, _ = s.draw(1, 0, 5)
    for q, x in zip(paths, w):
        assert abs(ref.score_of(q) - x) <= 1e-9 * abs(x)


@pytest.fixture(scope="module")
def fem(native_lib):
    from carmel_b200 import FOREST_CLI_PATH
    return FOREST_CLI_PATH


def test_sample_argument(fem, tmp_path):
    """--sample=n is refused with forest-em's argument-error exit (1, ERROR: ...) before any work: without -v, 0, a
    non-number, with --kbest, and with --shard / --gpus=N"""
    d = str(tmp_path)
    rng = np.random.default_rng(5)
    open(f"{d}/f", "w").write("\n".join(random_forest(rng, 10, depth=3) for _ in range(5)) + "\n")
    open(f"{d}/n", "w").write(random_normgroups(rng, 10))
    base = ["-f", f"{d}/f", "-n", f"{d}/n", "-i", "2"]
    for bad in ("0", "x", "-2", "", "3x"):
        rc, _, err = run(fem, [*base, "-v", f"{d}/v", f"--sample={bad}"])
        assert rc == 1 and "ERROR: --sample=n needs a whole number" in err, (bad, rc, err)
    rc, _, err = run(fem, [*base, "-v", f"{d}/v", "--sample"])
    assert rc == 1 and "ERROR: --sample=n needs a whole number" in err, err
    rc, _, err = run(fem, [*base, "--sample=3"])
    assert rc == 1 and "ERROR: --sample=n needs -v" in err, err
    for kb in ("--kbest=3", "--kbest=1"):
        rc, _, err = run(fem, [*base, "-v", f"{d}/v", "--sample=3", kb])
        assert rc == 1 and "ERROR: --sample=n draws derivations in place of --kbest" in err, err
    rc, _, err = run(fem, [*base, "-v", f"{d}/v", "--sample=3", "--shard=0/2"])
    assert rc == 1 and "ERROR: --sample draws on one GPU" in err, err
    rc, _, err = run(fem, [*base, "-v", f"{d}/v", "--sample=3", "--gpus=2"])
    assert rc == 1 and "ERROR: --sample draws on one GPU" in err, err
    assert not os.path.exists(f"{d}/v")
