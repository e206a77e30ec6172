"""k-best derivations of derivation forests on the GPU (cml_forests_kbest / k_forest_kbest, forest-em-b200 -v FILE
--kbest=n) against the CPU reference (forest_kbest_helpers.ForestRef: a lazy enumeration with a candidate heap per node)
under the comparison rule stated there; rank 0 against cml_forests_viterbi; chunking, determinism, depth and errors."""
import math

import numpy as np
import pytest

from forest_helpers import random_forest, random_normgroups, read_weights
from forest_kbest_helpers import compare_kbest, forest_refs, forests_to_arrays, read_kbest_forests
from helpers import run

pytestmark = pytest.mark.gpu
KS = (1, 2, 7, 32, 100)


def _forests(precision, n_rules):
    from carmel_b200.forest_api import Forests
    f = Forests(0, precision)
    f.set_rules(n_rules + 1, [0, n_rules], np.arange(1, n_rules + 1))
    return f


def _corpus(seed, n, n_rules, depth=5, share=0.2):
    rng = np.random.default_rng(seed)
    texts = [random_forest(rng, n_rules, depth=int(rng.integers(1, depth + 1)), share=share) for _ in range(n)]
    return texts, forests_to_arrays(texts), rng


def _got(score, n_and, base, nodes, i, k):
    return [(float(score[i, r]), tuple(int(x) for x in nodes[int(base[i * k + r]):int(base[i * k + r]) + int(n_and[i, r])]))
            for r in range(k)]


def _check(f, arrays, ln_w, ks=KS):
    refs = forest_refs(*arrays, ln_w)
    for k in ks:
        score, n_and, base, nodes = f.kbest(k, *arrays)
        assert score.shape == (len(refs), k)
        for i, ref in enumerate(refs):
            compare_kbest(ref.kbest(k), _got(score, n_and, base, nodes, i, k), ref.score_of)
        assert int(base[-1]) == int(n_and.sum())


@pytest.mark.parametrize("precision", [32, 64])
def test_kbest_against_reference(native_lib, precision):
    n_rules = 40
    texts, arrays, rng = _corpus(20271201 + precision, 60, n_rules)
    p = rng.uniform(0.05, 1.0, n_rules + 1)
    p[rng.random(n_rules + 1) < 0.1] = 0.0  # zero-weight rules
    with np.errstate(divide="ignore"):
        ln_w = np.log(p)
    f = _forests(precision, n_rules)
    f.set_params(ln_w)
    _check(f, arrays, ln_w)


@pytest.mark.parametrize("precision", [32, 64])
def test_kbest_ties(native_lib, precision):
    """exact ties: all weights one (ln 0, as -u -i 0 leaves them) and few, repeated rules with repeated weights"""
    n_rules = 3
    texts, arrays, rng = _corpus(20271301 + precision, 40, n_rules, depth=4, share=0.3)
    f = _forests(precision, n_rules)
    for ln_w in (np.zeros(n_rules + 1), np.log(np.array([1.0, 0.5, 0.5, 0.25]))):
        f.set_params(ln_w)
        _check(f, arrays, ln_w, ks=(1, 7, 32))


def _viterbi_nodes(nxt, label, backref, best, b, e):
    nx, lb, br, ch = nxt[b:e], label[b:e], backref[b:e], best[b:e]
    out = []

    def rec(c):
        while br[c] or lb[c] == 0:
            c = int(lb[c]) if br[c] else int(ch[c])
        out.append(c)
        q = c + 1
        while q < nx[c]:
            rec(q)
            q = int(nx[q])
    rec(0)
    return tuple(out)


def _rank0_is_viterbi(f, arrays, k=4):
    node_off, nxt, label, backref = arrays
    root, best = f.viterbi(*arrays)
    score, n_and, base, nodes = f.kbest(k, *arrays)
    finite = 0
    for i in range(len(node_off) - 1):
        if not root[i] > -math.inf:
            assert score[i, 0] == -math.inf
            continue
        finite += 1
        assert score[i, 0] == root[i], (i, score[i, 0], root[i])  # bit-identical
        got = tuple(int(x) for x in nodes[int(base[i * k]):int(base[i * k]) + int(n_and[i, 0])])
        assert got == _viterbi_nodes(nxt, label, backref, best, int(node_off[i]), int(node_off[i + 1])), i
    return finite


@pytest.mark.parametrize("precision", [32, 64])
def test_rank0_is_viterbi(native_lib, precision):
    n_rules = 30
    texts, arrays, rng = _corpus(20271401, 200, n_rules, depth=6)
    f = _forests(precision, n_rules)
    p = rng.choice([0.1, 0.2, 0.2, 0.5, 1.0], size=n_rules + 1)
    f.set_params(np.log(p))
    assert _rank0_is_viterbi(f, arrays) == 200


def test_rank0_is_viterbi_synthetic_corpus(native_lib):
    """a synth.make_forests batch of 3,000 forests: every forest's rank 0 is its Viterbi derivation"""
    from carmel_b200 import synth
    fs = synth.make_forests(n_forests=3000, n_rules=20000, templates=48, target_hyperedges=120)
    arrays = (fs["node_off"], fs["next"], fs["label"], fs["backref"])
    f = _forests(64, fs["n_rules"])
    rng = np.random.default_rng(5)
    f.set_params(np.log(rng.uniform(0.01, 1.0, fs["rulespace"])))
    assert _rank0_is_viterbi(f, arrays) == 3000


def test_chunking_and_determinism(native_lib):
    n_rules = 40
    texts, arrays, rng = _corpus(20271501, 120, n_rules)
    f = _forests(64, n_rules)
    f.set_params(np.log(rng.uniform(0.05, 1.0, n_rules + 1)))
    one = f.kbest(32, *arrays)
    assert f.kbest_stats()["chunks"] == 1
    again = f.kbest(32, *arrays)
    f.set_kbest_scratch_mb(1)
    split = f.kbest(32, *arrays)
    st = f.kbest_stats()
    assert st["chunks"] > 1 and st["scratch_bytes"] > 0, st
    for a, b, c in zip(one, again, split):
        assert a.tobytes() == b.tobytes() == c.tobytes()
    sizes = f.kbest(32, *arrays, nodes=False)
    for a, b in zip(one[:3], sizes[:3]):
        assert a.tobytes() == b.tobytes()


def test_deep_forest(native_lib):
    """200 nested levels with a shared node at each: cml_forests_viterbi keeps its 96-level error, k-best decodes"""
    from carmel_b200.api import CarmelB200Error
    body = "1"
    for d in range(200):
        body = f"(OR #{d + 1}(2 {body}) (3 #{d + 1}))"
    arrays = forests_to_arrays([body, "(OR 1 (2 3))"])
    ln_w = np.log(np.array([1.0, 0.5, 0.25, 0.75]))
    f = _forests(64, 3)
    f.set_params(ln_w)
    with pytest.raises(CarmelB200Error, match="deeper than 96"):
        f.viterbi(*arrays)
    _check(f, arrays, ln_w, ks=(1, 7, 32))


def test_errors(native_lib):
    import ctypes as C
    from carmel_b200.api import CarmelB200Error
    from carmel_b200.forest_api import _f64p, _u32p, _u64p
    texts, arrays, rng = _corpus(20271601, 10, 10)
    f = _forests(32, 10)
    with pytest.raises(CarmelB200Error) as e:  # before set_params
        f.kbest(3, *arrays)
    assert e.value.code == -3
    f.set_params(np.log(rng.uniform(0.1, 1.0, 11)))
    with pytest.raises(CarmelB200Error) as e:
        f.kbest(0, *arrays)
    assert e.value.code == -1
    # a node buffer that is too small: CML_ERR_ARG, with scores, sizes and bases still filled
    want = f.kbest(5, *arrays)
    b, keep = f._batch(*arrays)
    score, lens, base = np.empty(50), np.empty(50, np.uint32), np.zeros(51, np.uint64)
    small = np.empty(1, np.uint32)
    rc = f.lib.cml_forests_kbest(f.h, C.byref(b), 5, score.ctypes.data_as(_f64p), lens.ctypes.data_as(_u32p),
                                 base.ctypes.data_as(_u64p), small.ctypes.data_as(_u32p), 1)
    assert rc == -1 and int(base[-1]) > 1
    assert score.tobytes() == want[0].tobytes() and lens.tobytes() == want[1].tobytes() and base.tobytes() == want[2].tobytes()


@pytest.fixture(scope="module")
def fem(native_lib):
    from carmel_b200 import FOREST_CLI_PATH
    return FOREST_CLI_PATH


def test_cli_kbest(fem, tmp_path):
    """-v --kbest=n at the weights of 4 iterations of -U training against the reference; --kbest=1 is byte-identical to -v; the
    first line of every block is the -v line; padding lines read '0/<sum>=0% '"""
    rng = np.random.default_rng(20271701)
    d = str(tmp_path)
    texts = [random_forest(rng, n_rules=40, depth=5, share=0.2) for _ in range(60)] + ["(OR 1 2)", "(3 (OR 4 5))"]
    open(f"{d}/f", "w").write("\n".join(texts) + "\n")
    open(f"{d}/n", "w").write(random_normgroups(rng, 40, leave_out=0))
    rc, _, err = run(fem, ["-U", "-f", f"{d}/f", "-n", f"{d}/n", "-i", "4", "-o", f"{d}/w"])
    assert rc == 0, err
    # decode at the trained weights, read back (training's fp64 count sums are order-free up to the last bits, so two
    # training runs need not print the same digits; two decodes of the same weights must)
    args = ["-U", "-f", f"{d}/f", "-n", f"{d}/n", "-I", f"{d}/w", "-i", "0"]
    rc, _, err = run(fem, [*args, "-v", f"{d}/v1"])
    assert rc == 0, err
    rc, _, err = run(fem, [*args, "-v", f"{d}/vk1", "--kbest=1"])
    assert rc == 0, err
    assert open(f"{d}/v1", "rb").read() == open(f"{d}/vk1", "rb").read()
    k = 5
    rc, _, err = run(fem, [*args, "-v", f"{d}/vk", f"--kbest={k}"])
    assert rc == 0, err
    assert f"Viterbi: {k}-best lists, " in err
    lines, v1 = open(f"{d}/vk").read().split("\n")[:-1], open(f"{d}/v1").read().split("\n")[:-1]
    assert len(lines) == k * len(texts) and len(v1) == len(texts)
    got = read_kbest_forests(f"{d}/vk", k)
    ln_w = np.array([-math.inf] + read_weights(f"{d}/w"))
    refs = forest_refs(*forests_to_arrays(texts), ln_w)
    n_finite = 0
    for i, ref in enumerate(refs):
        if got[i][0][0] > -math.inf:
            n_finite += 1
            assert lines[i * k] == v1[i], (i, lines[i * k], v1[i])
        for r in range(k):
            if got[i][r][0] == -math.inf:
                assert lines[i * k + r].endswith("=0% ") and lines[i * k + r].startswith("0/"), lines[i * k + r]
        want = [(w, ref.tree(s) if s else "") for w, s in ref.kbest(k)]

        def run_of(r, ref=ref):
            m = 2 * k
            while True:
                lst = ref.kbest(m)
                s0 = lst[r][0]
                run_ = [ref.tree(s) for w, s in lst[r:] if w > -math.inf and abs(w - s0) <= 1e-12 * max(1.0, abs(s0))]
                if r + len(run_) < m or m >= 4096:
                    return run_
                m *= 2
        compare_kbest(want, [(w, t) for w, _, t in got[i]], run_of=run_of)
    assert n_finite > 30
    # the two small forests have 2 and 2 derivations: ranks 2..4 are padding
    for i in (len(texts) - 2, len(texts) - 1):
        assert [w > -math.inf for w, _, _ in got[i]] == [True, True, False, False, False]
