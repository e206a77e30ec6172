"""Decoding strings with the other tape free on the GPU (cml_build_free_trellises / k_build_free, carmel-b200 --decode):
the lattices against the CPU reference of decode_helpers.py array for array, the command line's k-best lists against
that reference under the comparison rule of kbest_helpers.py, consistency with the pair decoder (--viterbi) on cascades,
the tutorial's epron-jpron decode, and the C ABI's chunking, determinism and errors."""
import itertools
import math
import os
import re

import numpy as np
import pytest

import decode_helpers as D
from helpers import GOLDEN, run, sample_pairs, stage
from kbest_helpers import compare_kbest, read_kbest

pytestmark = pytest.mark.gpu
TAPE = {0: "input", 1: "output"}


def _cli(args, timeout=600):
    from carmel_b200 import CLI_PATH
    rc, _, err = run(CLI_PATH, args, timeout=timeout)
    assert rc == 0, err
    return err


def _decode(out, strings_file, model, given, k=None, extra=()):
    return _cli([f"--decode={out}", f"--given={TAPE[given]}", *(["-k", str(k)] if k else []), *extra, strings_file, *model])


def _random_strings(rng, names, n, max_len):
    return [" ".join(names[int(i)] for i in rng.integers(0, len(names), int(rng.integers(0, max_len + 1))))
            for _ in range(n)]


def _walks(m, given, rng, n, min_len):
    """n strings on tape `given` of random accepting walks of m, each at least min_len symbols long"""
    off, dst, lab, out = m["state_arc_off"], m["arc_dest"], (m["arc_in"], m["arc_out"])[given], []
    while len(out) < n:
        q, s = 0, []
        for _ in range(20 * min_len):
            if q == m["final_state"] and len(s) >= min_len:
                out.append(s)
                break
            if off[q] == off[q + 1]:
                break
            a = int(rng.integers(off[q], off[q + 1]))
            if lab[a]:
                s.append(int(lab[a]))
            q = int(dst[a])
    return out


def _check_cli(m, lines, given, path, k):
    """the --decode file at `path` against the reference under the comparison rule; every listed path a real
    derivation of its weight, its decoded-string column the free-tape labels of its arcs"""
    ids = [D.symbols(ln, m["alphabet"]) for ln in lines]
    want, lat, L = D.reference_kbest(m, ids, given, k)
    got = D.read_decode(path, k)
    assert len(got) == len(lines)
    lat_of = {int(e): i for i, e in enumerate(lat["kept"])}
    for e, (w, g) in enumerate(zip(want, got)):
        weight_of = (lambda p, i=lat_of[e]: L.weight(i, p)) if e in lat_of else (lambda p: None)
        compare_kbest([x[:2] for x in w], [x[:2] for x in g], weight_of)
        for gw, gp, gs in g:
            if gw > -math.inf:
                pw = weight_of(gp)
                assert pw is not None and abs(pw - gw) <= 1e-9 * max(1.0, abs(gw)), (e, gp, pw, gw)
                assert gs == D.decoded_string(m, gp, given), (e, gs)
            else:
                assert gp == () and gs == ""
    return want, got


def test_lattices_array_for_array(native_lib):
    """Context.build_free_trellises equals the reference builder array for array: 6 random machines and the golden
    epron-jpron.fst, both tapes, with empty, underivable and unknown-symbol strings"""
    from carmel_b200 import Context
    ctx = Context()
    cases = []
    for seed in range(6):
        rng = np.random.default_rng(20271301 + seed)
        m, _ = D.random_machine(rng, n_states=int(rng.integers(2, 7)), eps_rate=float(rng.uniform(0.1, 0.4)))
        for given, (lo, hi) in ((0, (1, 4)), (1, (4, 7))):
            strings = [[int(x) for x in rng.integers(lo, hi, int(rng.integers(0, 7)))] for _ in range(40)]
            cases.append((m, strings + [[], [lo, 77], [0], [hi + 5]], given))
    g = D.parse_wfst(open(os.path.join(GOLDEN, "epron-jpron.fst")).read())
    data = open(os.path.join(GOLDEN, "epron-jpron.data")).read().splitlines()
    for given in (0, 1):
        strings = [D.symbols(ln, g["alphabet"]) for ln in data[given::2]]
        cases.append((g, strings + [[], D.symbols('"no-such-symbol"', g["alphabet"])], given))
    n_kept = 0
    for m, strings, given in cases:
        got = ctx.build_free_trellises(m, strings, given)
        want = D.free_lattices(m, strings, given)
        assert got["n_ex"] == want["n_ex"]
        for key in ("ex_states", "ex_fin", "arc_off", "arc_dst", "arc_id", "kept", "dropped"):
            assert np.array_equal(got[key], want[key]), key
        assert np.all(got["ex_weight"] == 1.0)
        n_kept += want["n_ex"]
    assert n_kept > 30


@pytest.mark.parametrize("trained", [False, True])
@pytest.mark.parametrize("given", [0, 1])
def test_cli_against_reference(native_lib, oracle_bin, tmp_path, given, trained):
    """carmel-b200 --decode -k {1, 5, 50} against the reference lists; rank 0 of -k n is the -k 1 file byte for byte"""
    for seed in range(3):
        rng = np.random.default_rng(20271401 + 10 * seed + given)
        ns = int(rng.integers(2, 6))
        m0, text = D.random_machine(rng, n_states=ns, eps_rate=float(rng.uniform(0.1, 0.4)))
        d = str(tmp_path / f"s{seed}")
        os.makedirs(d)
        fst = os.path.join(d, "m.fst")
        open(fst, "w").write(text)
        if trained:
            names = m0["names"]
            arcs = [(s, int(m0["arc_dest"][a]), names[int(m0["arc_in"][a])] if m0["arc_in"][a] else None,
                     names[int(m0["arc_out"][a])] if m0["arc_out"][a] else None)
                    for s in range(ns) for a in range(m0["state_arc_off"][s], m0["state_arc_off"][s + 1])]
            open(os.path.join(d, "c.data"), "w").write(sample_pairs(rng, arcs, ns, n_pairs=10, max_steps=6))
            _cli(["-t", "-F", os.path.join(d, "trained.fst"), os.path.join(d, "c.data"), fst])
            fst = os.path.join(d, "trained.fst")
        given_names = [f'"{"io"[given]}{j}"' for j in range(3)]
        lines = _random_strings(rng, given_names, 14, 4) + ['"zz"', ""]
        sf = os.path.join(d, "s.txt")
        open(sf, "w").write("\n".join(lines) + "\n")
        m = D.reference_model(oracle_bin, d, [fst])
        err = _decode(os.path.join(d, "k1"), sf, [fst], given)
        assert f"Decode: {len(lines)} strings on the {TAPE[given]} tape" in err, err
        one = open(os.path.join(d, "k1")).read().splitlines()
        assert len(one) == len(lines)
        _check_cli(m, lines, given, os.path.join(d, "k1"), 1)
        for k in (5, 50):
            p = os.path.join(d, f"k{k}")
            err = _decode(p, sf, [fst], given, k)
            assert f"Decode: {k}-best lists" in err, err
            _check_cli(m, lines, given, p, k)
            many = open(p).read().splitlines()
            assert [many[e * k] for e in range(len(lines))] == one
            assert len(read_kbest(p, k)) == len(lines)  # the --viterbi reader still parses the file


def _viterbi_pairs(d, pairs, model, k=None):
    """--viterbi on (input, output) pairs: per pair the list of (ln weight) of its k best derivations, None when the pair
    has no derivation"""
    c = os.path.join(d, "pairs.data")
    open(c, "w").write("".join(f"{a}\n{b}\n" for a, b in pairs))
    out = os.path.join(d, "pairs.v")
    err = _cli([f"--viterbi={out}", *(["-k", str(k)] if k else []), c, *model])
    dropped = {int(x) - 1 for x in re.findall(r"No derivations in transducer for input/output #(\d+)", err)}
    lines = open(out).read().splitlines()
    kk = k or 1
    res, i = [], 0
    for e in range(len(pairs)):
        if e in dropped:
            res.append(None)
            continue
        res.append([float(ln.split()[0]) for ln in lines[i * kk:(i + 1) * kk]])
        i += 1
    assert i * kk == len(lines)
    return res


@pytest.mark.parametrize("given", [0, 1])
@pytest.mark.parametrize("seed", range(3))
def test_cascades_agree_with_the_pair_decoder(native_lib, oracle_bin, tmp_path, seed, given):
    """2-member random cascades (--train-cascade): every best string x* decoded for s has, as the pair (x*, s) on
    --viterbi, the same ln weight (1e-12 relative); and over all free strings up to the lattice's longest path, the top
    k of the union of their --viterbi -k k lists are the free decode's k weights (1e-9)"""
    rng = np.random.default_rng(20271501 + 10 * seed + given)
    d = str(tmp_path)
    a, b = os.path.join(d, "a.fst"), os.path.join(d, "b.fst")
    model = ["--train-cascade", a, b]
    for _ in range(50):  # draw until the two members compose to a non-empty machine
        _, ta = D.random_machine(rng, n_states=int(rng.integers(2, 4)), n_in=2, n_out=2, eps_rate=0.2, out_prefix="m")
        _, tb = D.random_machine(rng, n_states=int(rng.integers(2, 4)), n_in=2, n_out=2, eps_rate=0.2, in_prefix="m")
        open(a, "w").write(ta)
        open(b, "w").write(tb)
        open(os.path.join(d, "empty.data"), "w").close()
        if run(oracle_bin, ["--train-cascade", f"--dump-estimate={d}/e", os.path.join(d, "empty.data"), a, b])[0] == 0:
            break
    names = [f'"{"io"[given]}{j}"' for j in range(2)]
    lines = [" ".join(p) for n in range(3) for p in itertools.product(names, repeat=n)]
    sf = os.path.join(d, "s.txt")
    open(sf, "w").write("\n".join(lines) + "\n")
    k = 4
    _decode(os.path.join(d, "dec"), sf, model, given, k)
    got = D.read_decode(os.path.join(d, "dec"), k)
    found = [e for e in range(len(lines)) if got[e][0][0] > -math.inf]
    assert found, "no string has a derivation"
    pair = lambda s, x: (x, s) if given == 1 else (s, x)
    best = _viterbi_pairs(d, [pair(lines[e], got[e][0][2]) for e in found], model)
    for e, v in zip(found, best):
        assert v is not None and abs(v[0] - got[e][0][0]) <= 1e-12 * max(1.0, abs(v[0])), (e, v, got[e][0])
    # exhaustive: the free decode's k weights are the top k over every free string's pair derivations
    m = D.reference_model(oracle_bin, d, model)
    lat = D.free_lattices(m, [D.symbols(ln, m["alphabet"]) for ln in lines], given)
    free = m["arc_out"] if given == 0 else m["arc_in"]
    alphabet = sorted({m["names"][int(x)] for x in free if x})
    checked = 0
    for i, e in enumerate(lat["kept"]):
        bound = D.longest_path(lat, i)
        if len(alphabet) ** bound > 2000:
            continue
        xs = [" ".join(p) for n in range(bound + 1) for p in itertools.product(alphabet, repeat=n)]
        lists = _viterbi_pairs(d, [pair(lines[e], x) for x in xs], model, k)
        union = sorted((w for v in lists if v for w in v if w > -math.inf), reverse=True)
        top = (union + [-math.inf] * k)[:k]
        for r, (tw, (gw, _, _)) in enumerate(zip(top, got[e])):
            assert tw == gw == -math.inf or abs(tw - gw) <= 1e-9 * max(1.0, abs(tw)), (e, r, tw, gw)
        checked += 1
    assert checked >= 1


def test_tagging_agrees_with_the_pair_decoder(native_lib, tmp_path):
    """the tagging shape with the tags on the free tape: a tag:tag bigram (tagging.fsa with each *e*:tag arc made
    tag:tag) o tagging.fst, the words given; each best tag sequence as a pair on --viterbi has the same ln weight"""
    d = str(tmp_path)
    src, fst = stage(tmp_path, "tagging.data", "tagging.fst")
    fsa = os.path.join(d, "tags.fsa")
    open(fsa, "w").write(re.sub(r'\*e\* ("[^"]*")', r"\1 \1", open(os.path.join(GOLDEN, "tagging.fsa")).read()))
    sents = open(src).read().splitlines()[1::2][:12]
    sf = os.path.join(d, "s.txt")
    open(sf, "w").write("\n".join(sents) + "\n")
    model = ["--train-cascade", fsa, fst]
    _decode(os.path.join(d, "dec"), sf, model, 1)
    got = D.read_decode(os.path.join(d, "dec"), 1)
    found = [e for e in range(len(sents)) if got[e][0][0] > -math.inf]
    assert len(found) >= 6
    best = _viterbi_pairs(d, [(got[e][0][2], sents[e]) for e in found], model)
    for e, v in zip(found, best):
        assert v is not None and abs(v[0] - got[e][0][0]) <= 1e-12 * max(1.0, abs(v[0])), (e, v, got[e][0])


def test_epron_jpron_tutorial_decode(native_lib, oracle_bin, tmp_path):
    """train epron-jpron.fst on its pairs, then decode each pair's Japanese side with --given=output -k 5: the lists
    match the reference, and the pair's own English side is among the 5 best decoded strings"""
    d = str(tmp_path)
    data, fst = stage(tmp_path, "epron-jpron.data", "epron-jpron.fst")
    trained = os.path.join(d, "epron-jpron.fst.trained")
    _cli(["-t", "-F", trained, data, fst])
    pairs = open(data).read().splitlines()
    eng, jp = pairs[0::2], pairs[1::2]
    sf = os.path.join(d, "jpron.txt")
    open(sf, "w").write("\n".join(jp) + "\n")
    out = os.path.join(d, "out")
    _decode(out, sf, [trained], 1, 5)
    lines = open(out).read().splitlines()
    assert len(lines) == 5 * len(jp)
    for e in range(len(jp)):  # each line ends in a decoded English string, or pads a list of fewer than 5 derivations
        ranks = lines[5 * e:5 * e + 5]
        n = sum(1 for ln in ranks if re.search(r' \|\| \S', ln))
        assert all(ln == "-inf 0 | ||" for ln in ranks[n:]), ranks
    m = D.reference_model(oracle_bin, d, [trained])
    _, got = _check_cli(m, jp, 1, out, 5)
    for e, x in enumerate(eng):
        assert " ".join(x.split()) in [g[2] for g in got[e]], (x, got[e])


def test_chunks_determinism_and_errors(native_lib, tmp_path):
    from carmel_b200 import api as cb
    ctx = cb.Context()
    g = D.parse_wfst(open(os.path.join(GOLDEN, "epron-jpron.fst")).read())
    rng = np.random.default_rng(20271601)
    strings = _walks(g, 1, rng, 300, 20) + [[int(x) for x in rng.choice(g["arc_out"], 30)] for _ in range(20)]
    one = ctx.build_free_trellises(g, strings, 1)
    assert one["stats"]["chunks"] == 1 and one["n_ex"] > 100
    again = ctx.build_free_trellises(g, strings, 1)
    ctx.set_option(cb.OPT_FREE_BUILD_SCRATCH_MB, 1)
    split = ctx.build_free_trellises(g, strings, 1)
    assert split["stats"]["chunks"] > 2
    for other in (again, split):
        for key in ("ex_states", "ex_fin", "arc_off", "arc_dst", "arc_id", "kept", "dropped"):
            assert one[key].tobytes() == other[key].tobytes(), key
    # a given-*e* cycle: CML_ERR_CYCLE from the C ABI, exit -11 from the command line
    m = dict(n_states=3, final_state=2, state_arc_off=np.array([0, 1, 3, 3], np.uint32), arc_in=np.array([1, 2, 1], np.uint32),
             arc_out=np.array([0, 0, 3], np.uint32), arc_dest=np.array([1, 0, 2], np.uint32))
    assert ctx.build_free_trellises(m, [[1, 1]], 0)["n_ex"] == 1
    with pytest.raises(cb.CarmelB200Error) as ex:
        ctx.build_free_trellises(m, [[3]], 1)
    assert ex.value.code == cb.ERR_CYCLE
    f, sf = os.path.join(str(tmp_path), "c.fst"), os.path.join(str(tmp_path), "s.txt")
    open(f, "w").write('q2\n(q0 (q1 "a" *e* 0.5))\n(q1 (q0 "b" *e* 0.5))\n(q1 (q2 "a" "x" 0.5))\n')
    open(sf, "w").write('"x"\n')
    from carmel_b200 import CLI_PATH
    rc, _, err = run(CLI_PATH, [f"--decode={tmp_path}/o", "--given=output", sf, f])
    assert rc == -11 % 256 and "ERROR:" in err and "form a cycle" in err, (rc, err)
    # CML_ERR_ARG: a bad tape, offsets that decrease or do not start at 0
    for strs, tape in (([[1]], 2), (([0, 2, 1], [1, 1]), 0), (([1, 2], [1, 1]), 0)):
        with pytest.raises(cb.CarmelB200Error) as ex:
            ctx.build_free_trellises(m, strs, tape)
        assert ex.value.code == cb.ERR_ARG
