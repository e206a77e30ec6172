"""Sums and samples of derivation forests on the GPU (cml_forests_sample / k_forest_sample, forest-em-b200 -v FILE
--sample=n) against the CPU reference (forest_sample_helpers.ForestSampler: memoised inside recursion, a recursive walk
per sample) under the comparison rule stated there; the GPU's own draws by chi-square; keys, chunking, determinism,
depth, the size refusal, the error codes and the command line."""
import math
import time

import numpy as np
import pytest

from forest_helpers import random_forest, random_normgroups, read_weights
from forest_kbest_helpers import ForestRef, forests_to_arrays, read_kbest_forests
from forest_sample_helpers import EXEMPT_SHARE, chi2_fit, compare_samples, forest_samplers, small_forests
from helpers import run

pytestmark = pytest.mark.gpu


def _forests(precision, n_rules):
    from carmel_b200.forest_api import Forests
    f = Forests(0, precision)
    f.set_rules(n_rules + 1, [0, n_rules], np.arange(1, n_rules + 1))
    return f


def _corpus(seed, n, n_rules, depth=5, share=0.2):
    rng = np.random.default_rng(seed)
    texts = [random_forest(rng, n_rules, depth=int(rng.integers(1, depth + 1)), share=share) for _ in range(n)]
    return texts, forests_to_arrays(texts), rng


def _got(lnw, n_and, base, nodes, i, n):
    return [(float(lnw[i, r]), tuple(int(x) for x in nodes[int(base[i * n + r]):int(base[i * n + r]) + int(n_and[i, r])]))
            for r in range(n)]


def _check(f, arrays, ln_w, ns=(1, 7, 100), seed=11, key=None):
    samplers = forest_samplers(*arrays, ln_w)
    for n in ns:
        lnw, n_and, base, nodes, total = f.sample(n, seed, *arrays, key=key)
        assert lnw.shape == (len(samplers), n)
        n_ex = 0
        for i, s in enumerate(samplers):
            k = i if key is None else int(key[i])
            n_ex += compare_samples(s, s.draw(seed, k, n), float(total[i]), _got(lnw, n_and, base, nodes, i, n))
        assert n_ex <= EXEMPT_SHARE * n * len(samplers), (n, n_ex)
        assert int(base[-1]) == int(n_and.sum())


@pytest.mark.parametrize("precision", [32, 64])
def test_sample_against_reference(native_lib, precision):
    n_rules = 40
    texts, arrays, rng = _corpus(20281301 + precision, 60, n_rules)
    p = rng.uniform(0.05, 1.0, n_rules + 1)
    p[rng.random(n_rules + 1) < 0.1] = 0.0  # zero-weight rules
    with np.errstate(divide="ignore"):
        ln_w = np.log(p)
    f = _forests(precision, n_rules)
    f.set_params(ln_w)
    _check(f, arrays, ln_w)


@pytest.mark.parametrize("precision", [32, 64])
def test_sample_ties(native_lib, precision):
    """exact ties: all weights one (ln 0) and few, repeated rules with repeated weights"""
    n_rules = 3
    texts, arrays, rng = _corpus(20281401 + precision, 40, n_rules, depth=4, share=0.3)
    f = _forests(precision, n_rules)
    for ln_w in (np.zeros(n_rules + 1), np.log(np.array([1.0, 0.5, 0.5, 0.25]))):
        f.set_params(ln_w)
        _check(f, arrays, ln_w, ns=(1, 7))


def test_totals_only_and_against_the_estep(native_lib):
    """n = 0 gives ln_total only (the same values as with n > 0); on an fp64 handle ln_total agrees with the E-step's
    inside values to 1e-10 relative"""
    n_rules = 30
    texts, arrays, rng = _corpus(20281501, 80, n_rules)
    ln_w = np.log(rng.uniform(0.05, 1.0, n_rules + 1))
    f = _forests(64, n_rules)
    f.set_params(ln_w)
    f.add(*arrays)
    f.estimate()
    ins = f.inside(80)
    lnw, n_and, base, nodes, total = f.sample(0, 3, *arrays)
    assert lnw.shape == (80, 0) and nodes is None and len(base) == 1
    assert total.tobytes() == f.sample(5, 3, *arrays)[4].tobytes()
    for i in range(80):
        assert abs(total[i] - ins[i]) <= 1e-10 * max(1.0, abs(ins[i])), (i, total[i], ins[i])
    assert f.sample_stats()["kernel_ms"] > 0


def test_gpu_draws_chi_square(native_lib):
    """the GPU's own draws: 20 small forests (shared nodes, zero-weight rules), 20,000 samples each at a fixed seed"""
    rng = np.random.default_rng(20281601)
    n_rules = 10
    p = rng.choice([0.0, 0.25, 0.5, 1.0, 0.125, 0.9], size=n_rules + 1)
    with np.errstate(divide="ignore"):
        ln_w = np.log(p)
    texts = []
    for t in small_forests(rng, 400, n_rules):
        s = forest_samplers(*forests_to_arrays([t]), ln_w)[0]
        if s.ln_total() > -math.inf and len(s.derivations()) >= 2:
            texts.append(t)
        if len(texts) == 20:
            break
    assert len(texts) == 20
    arrays = forests_to_arrays(texts)
    f = _forests(64, n_rules)
    f.set_params(ln_w)
    n = 20000
    lnw, n_and, base, nodes, total = f.sample(n, 20281602, *arrays)
    for i, s in enumerate(forest_samplers(*arrays, ln_w)):
        paths = [q for _, q in _got(lnw, n_and, base, nodes, i, n)]
        assert chi2_fit(s, paths) > 1e-6, (i, texts[i])


def test_key(native_lib):
    """forest i drawn alone with key=[i] equals forest i drawn inside the batch; explicit keys follow the reference"""
    n_rules = 20
    texts, arrays, rng = _corpus(20281701, 30, n_rules)
    ln_w = np.log(rng.uniform(0.05, 1.0, n_rules + 1))
    f = _forests(64, n_rules)
    f.set_params(ln_w)
    n = 9
    lnw, n_and, base, nodes, total = f.sample(n, 5, *arrays)
    for i in (0, 7, 29):
        one = forests_to_arrays([texts[i]])
        l1, z1, b1, x1, t1 = f.sample(n, 5, *one, key=[i])
        assert l1.tobytes() == lnw[i:i + 1].tobytes() and z1.tobytes() == n_and[i:i + 1].tobytes()
        assert t1.tobytes() == total[i:i + 1].tobytes()
        assert x1.tobytes() == nodes[int(base[i * n]):int(base[i * n + n])].tobytes()
    _check(f, arrays, ln_w, ns=(7,), key=rng.integers(0, 2 ** 63, 30, dtype=np.uint64))


def test_chunking_and_determinism(native_lib):
    n_rules = 40
    texts, arrays, rng = _corpus(20281801, 150, n_rules)
    f = _forests(64, n_rules)
    f.set_params(np.log(rng.uniform(0.05, 1.0, n_rules + 1)))
    one = f.sample(100, 9, *arrays)
    assert f.sample_stats()["chunks"] == 1
    again = f.sample(100, 9, *arrays)
    f.set_kbest_scratch_mb(1)
    split = f.sample(100, 9, *arrays)
    st = f.sample_stats()
    assert st["chunks"] > 1 and st["scratch_bytes"] > 0, st
    for a, b, c in zip(one, again, split):
        assert a.tobytes() == b.tobytes() == c.tobytes()
    sizes = f.sample(100, 9, *arrays, nodes=False)
    assert sizes[3] is None
    for i in (0, 1, 2, 4):
        assert one[i].tobytes() == sizes[i].tobytes()


def test_deep_forest(native_lib):
    """200 nested levels with a shared node at each (cml_forests_viterbi refuses it at 96 levels): samples"""
    body = "1"
    for d in range(200):
        body = f"(OR #{d + 1}(2 {body}) (3 #{d + 1}))"
    arrays = forests_to_arrays([body, "(OR 1 (2 3))"])
    ln_w = np.log(np.array([1.0, 0.5, 0.25, 0.75]))
    f = _forests(64, 3)
    f.set_params(ln_w)
    _check(f, arrays, ln_w, ns=(1, 7, 100))


def test_doubling_forest_is_refused(native_lib):
    """a forest whose derivation doubles at each of 40 levels (about 2^41 AND nodes) returns CML_ERR_ARG promptly; its
    total is still computed with n = 0"""
    from carmel_b200.api import CarmelB200Error
    body = "#1(2 3)"
    for d in range(40):
        body = f"#{d + 2}(1 {body} #{d + 1})"
    arrays = forests_to_arrays([body])
    f = _forests(64, 3)
    f.set_params(np.log(np.array([1.0, 0.5, 0.25, 0.75])))
    t0 = time.perf_counter()
    with pytest.raises(CarmelB200Error, match="more than 2\\^32 - 2 AND nodes") as e:
        f.sample(3, 1, *arrays)
    assert e.value.code == -1 and time.perf_counter() - t0 < 30
    assert math.isfinite(f.sample(0, 1, *arrays)[4][0])


def test_errors(native_lib):
    import ctypes as C
    from carmel_b200.api import CarmelB200Error
    from carmel_b200.forest_api import _f64p, _u32p, _u64p
    texts, arrays, rng = _corpus(20281901, 10, 10)
    f = _forests(32, 10)
    with pytest.raises(CarmelB200Error) as e:  # before set_params
        f.sample(3, 1, *arrays)
    assert e.value.code == -3
    f.set_params(np.log(rng.uniform(0.1, 1.0, 11)))
    b, keep = f._batch(*arrays)
    lnw, lens, base, tot = np.empty(50), np.empty(50, np.uint32), np.zeros(51, np.uint64), np.empty(10)
    P = lambda a, t: a.ctypes.data_as(t)
    assert f.lib.cml_forests_sample(f.h, C.byref(b), 5, 1, None, P(lnw, _f64p), P(lens, _u32p), P(base, _u64p), None, 0,
                                    None) == -1  # null ln_total
    assert f.lib.cml_forests_sample(f.h, C.byref(b), 5, 1, None, None, P(lens, _u32p), P(base, _u64p), None, 0,
                                    P(tot, _f64p)) == -1  # n > 0, null ln_weight
    # a node buffer that is too small: CML_ERR_ARG, with weights, sizes, bases and totals still filled
    want = f.sample(5, 1, *arrays)
    small = np.empty(1, np.uint32)
    rc = f.lib.cml_forests_sample(f.h, C.byref(b), 5, 1, None, P(lnw, _f64p), P(lens, _u32p), P(base, _u64p),
                                  P(small, _u32p), 1, P(tot, _f64p))
    assert rc == -1 and int(base[-1]) > 1
    assert lnw.tobytes() == want[0].tobytes() and lens.tobytes() == want[1].tobytes()
    assert base.tobytes() == want[2].tobytes() and tot.tobytes() == want[4].tobytes()
    # a rule id beyond rulespace, a malformed forest (an OR node without children)
    with pytest.raises(CarmelB200Error) as e:
        f.sample(2, 1, *forests_to_arrays(["(OR 1 99)"]))
    assert e.value.code == -1 and "beyond rulespace" in str(e.value)
    bad = (np.array([0, 2], np.uint64), np.array([2, 2], np.uint32), np.array([0, 0], np.uint32), np.array([0, 0], np.uint8))
    with pytest.raises(CarmelB200Error) as e:
        f.sample(2, 1, *bad)
    assert e.value.code == -1 and "malformed" in str(e.value)


def test_cycle(native_lib):
    """CML_ERR_CYCLE for a back reference to an ancestor, as cml_forests_kbest reports it"""
    from carmel_b200.api import CarmelB200Error
    # pre-order: 0 = OR (root), 1 = AND rule 1 defining #1, 2 = OR under it, 3 = leaf 2, 4 = backref to node 1
    arrays = (np.array([0, 5], np.uint64), np.array([5, 5, 5, 4, 5], np.uint32), np.array([0, 1, 0, 2, 1], np.uint32),
              np.array([0, 0, 0, 0, 1], np.uint8))
    f = _forests(64, 3)
    f.set_params(np.zeros(4))
    with pytest.raises(CarmelB200Error) as ek:
        f.kbest(2, *arrays)
    with pytest.raises(CarmelB200Error) as es:
        f.sample(2, 1, *arrays)
    assert es.value.code == ek.value.code == -4


@pytest.fixture(scope="module")
def fem(native_lib):
    from carmel_b200 import FOREST_CLI_PATH
    return FOREST_CLI_PATH


def test_cli_sample(fem, tmp_path):
    """-v --sample=n at the weights of 4 iterations of -U training: n lines per forest, every line the reference's draw
    under the rule (trees compared as text), padding lines '0/<sum>=0% ' for zero-probability forests, the same file
    from two runs and a different one for another --seed"""
    rng = np.random.default_rng(20282001)
    d = str(tmp_path)
    texts = [random_forest(rng, n_rules=40, depth=5, share=0.2) for _ in range(60)] + ["(OR 1 2)", "(3 (OR 4 5))"]
    open(f"{d}/f", "w").write("\n".join(texts) + "\n")
    open(f"{d}/n", "w").write(random_normgroups(rng, 40, leave_out=0))
    rc, _, err = run(fem, ["-U", "-f", f"{d}/f", "-n", f"{d}/n", "-i", "4", "-o", f"{d}/w"])
    assert rc == 0, err
    ln_w = np.array([-math.inf] + read_weights(f"{d}/w"))
    # a zero-probability forest: rule 41 gets weight zero in a copy of the trained weights
    texts.append("(OR (41 1) (2 41))")
    open(f"{d}/f", "w").write("\n".join(texts) + "\n")
    open(f"{d}/w0", "w").write(open(f"{d}/w").read().rstrip("\n") + " 0\n")
    groups = open(f"{d}/n").read().strip()
    open(f"{d}/n", "w").write(groups[:-1] + " (41))\n")
    ln_w = np.append(ln_w, -math.inf)
    args = ["-U", "-f", f"{d}/f", "-n", f"{d}/n", "-I", f"{d}/w0", "-i", "0"]
    n = 5
    for name, seed in (("s1", 7), ("s2", 7), ("s3", 8)):
        rc, _, err = run(fem, [*args, "-v", f"{d}/{name}", f"--sample={n}", f"--seed={seed}"])
        assert rc == 0, err
    assert f"Viterbi: {n} samples per forest, " in err
    assert open(f"{d}/s1", "rb").read() == open(f"{d}/s2", "rb").read()
    assert open(f"{d}/s1", "rb").read() != open(f"{d}/s3", "rb").read()
    lines = open(f"{d}/s1").read().split("\n")[:-1]
    assert len(lines) == n * len(texts)
    got = read_kbest_forests(f"{d}/s1", n)
    arrays = forests_to_arrays(texts)
    samplers = forest_samplers(*arrays, ln_w)
    n_ex = 0
    for i, s in enumerate(samplers):
        ref = ForestRef(arrays[1][int(arrays[0][i]):int(arrays[0][i + 1])], arrays[2][int(arrays[0][i]):int(arrays[0][i + 1])],
                        arrays[3][int(arrays[0][i]):int(arrays[0][i + 1])], ln_w)
        paths, w, ex = s.draw(7, i, n)
        if s.ln_total() == -math.inf:
            for r in range(n):
                assert lines[i * n + r].startswith("0/") and lines[i * n + r].endswith("=0% "), lines[i * n + r]
            continue
        for r in range(n):
            gw, _, tree = got[i][r]
            if ex[r] >= 0:
                n_ex += 1
                continue
            assert tree == ref.tree(paths[r]), (i, r, tree, ref.tree(paths[r]))
            assert abs(gw - w[r]) <= 1e-9 * max(1.0, abs(w[r])), (i, r, gw, w[r])  # printed with limited digits
    assert n_ex <= max(1, EXEMPT_SHARE * n * len(texts))
    assert samplers[-1].ln_total() == -math.inf
