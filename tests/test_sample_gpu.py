"""Sums and samples on the GPU (cml_sample / k_sample, carmel-b200 --sum / --sample) against the CPU reference of
sample_helpers.py: ln totals to 1e-12, draws under its comparison rule, the distribution under its chi-square rule, the
free-string sums against the pair sums of every free string, the command line, and the C ABI's chunking, determinism and
errors."""
import itertools
import math
import os

import numpy as np
import pytest

import decode_helpers as D
import sample_helpers as S
from helpers import GOLDEN, random_wfst, read_estimate_dump, read_trellis_dump, run, sample_pairs, stage
from kbest_helpers import Lattices, read_kbest

pytestmark = pytest.mark.gpu
TAPE = {0: "input", 1: "output"}


def _cli(args, timeout=600):
    from carmel_b200 import CLI_PATH
    rc, _, err = run(CLI_PATH, args, timeout=timeout)
    assert rc == 0, err
    return err


def _close(a, b, rel=1e-12):
    return a == b or abs(a - b) <= rel * max(1.0, abs(a), abs(b))


def _rows(ln_w, lens, base, arcs):
    n_ex, n = lens.shape
    return [[(float(ln_w[e, r]), tuple(int(x) for x in arcs[base[e * n + r]:base[e * n + r] + lens[e, r]]))
             for r in range(n)] for e in range(n_ex)]


def _check_lattice(smp, e, got_total, got, seed, key):
    """ln total, and the draws under the comparison rule; every drawn path a real derivation of its weight.  Returns
    the number of exempt samples."""
    want_total = smp.ln_total(e)
    assert (want_total == -math.inf and got_total == -math.inf) or _close(want_total, got_total), (e, want_total, got_total)
    n_ex = S.compare_draws(smp.draw(e, seed, key, len(got)), got)
    for w, p in got:
        if want_total == -math.inf:
            assert w == -math.inf and p == ()
        else:
            pw = smp.L.weight(e, p)
            assert pw is not None and _close(pw, w), (e, p, pw, w)
    return n_ex


def _pairs_case(oracle_bin, d, args, n=200, seed=5):
    """--no-ell job on the pair lattices of `args`: sums and draws against the reference over the oracle's lattices,
    and ln totals against the E-step's per-example ln P on the same context"""
    from carmel_b200 import Job
    rc, _, err = run(oracle_bin, [f"--dump-trellis={d}/t", f"--dump-estimate={d}/e", *args], timeout=600)
    assert rc == 0, err
    lat = Lattices(read_trellis_dump(f"{d}/t"), read_estimate_dump(f"{d}/e")["ln_w"])
    smp = S.Sampler(lat)
    job = Job(["--no-ell", "--no-dense", "--no-lane", *args])
    ctx = job.prepare()
    tot, w, ln, b, a = ctx.sample(n, seed)
    tot0 = ctx.sample(0, seed)[0]
    assert tot.tobytes() == tot0.tobytes()
    got = _rows(w, ln, b, a)
    assert len(got) == lat.t["n_ex"]
    exempt = sum(_check_lattice(smp, e, tot[e], got[e], seed, e) for e in range(len(got)))
    assert exempt <= 0.001 * n * len(got), exempt
    ctx.estimate()
    lnp = ctx.example_logprob(len(got))
    for e in range(len(got)):
        assert _close(float(lnp[e]), float(tot[e])), (e, lnp[e], tot[e])
    job.close()
    return tot


@pytest.mark.parametrize("seed", range(4))
def test_pairs_random_transducers(native_lib, oracle_bin, tmp_path, seed):
    rng = np.random.default_rng(20271901 + seed)
    ns = int(rng.integers(2, 7))
    fst, ins, outs, arcs = random_wfst(rng, n_states=ns, eps_rate=float(rng.uniform(0, 0.4)))
    d = str(tmp_path)
    open(f"{d}/r.fst", "w").write(fst)
    open(f"{d}/r.data", "w").write(sample_pairs(rng, arcs, ns, n_pairs=12, max_steps=7, ins=ins, outs=outs))
    _pairs_case(oracle_bin, d, ["-t", f"{d}/r.data", f"{d}/r.fst"], seed=seed + 1)


@pytest.mark.parametrize("trained", [True, False])
def test_pairs_cipher(native_lib, oracle_bin, tmp_path, trained):
    data, wfsa = stage(tmp_path, "cipher.data", "cipher.wfsa")
    fst = os.path.join(str(tmp_path), "cipher.fst")
    open(fst, "w").write(open(os.path.join(GOLDEN, "cipher.fst.trained" if trained else "cipher.fst")).read())
    _pairs_case(oracle_bin, str(tmp_path), ["--train-cascade", data, wfsa, fst], n=300)


def test_pairs_tagging(native_lib, oracle_bin, tmp_path):
    src, fsa, fst = stage(tmp_path, "tagging.data", "tagging.fsa", "tagging.fst")
    data = os.path.join(str(tmp_path), "t20.data")
    open(data, "w").write("".join(open(src).readlines()[:40]))
    _pairs_case(oracle_bin, str(tmp_path), ["--train-cascade", data, fsa, fst], n=300)


@pytest.mark.parametrize("given", [0, 1])
def test_free_strings_cli(native_lib, oracle_bin, tmp_path, given):
    """--decode --sum / --sample on random machines: sums and draws against the reference on free_lattices (keys = the
    string's line); adding --sum leaves the 5-best file unchanged"""
    n = 100
    for seed in range(3):
        rng = np.random.default_rng(20272001 + 10 * seed + given)
        m0, text = D.random_machine(rng, n_states=int(rng.integers(2, 6)), eps_rate=float(rng.uniform(0.1, 0.4)))
        d = str(tmp_path / f"s{seed}")
        os.makedirs(d)
        fst = os.path.join(d, "m.fst")
        open(fst, "w").write(text)
        names = [f'"{"io"[given]}{j}"' for j in range(3)]
        lines = [" ".join(names[int(i)] for i in rng.integers(0, 3, int(rng.integers(0, 5)))) for _ in range(14)]
        lines += ['"zz"', ""]
        sf = os.path.join(d, "s.txt")
        open(sf, "w").write("\n".join(lines) + "\n")
        m = D.reference_model(oracle_bin, d, [fst])
        lat = D.free_lattices(m, [D.symbols(ln, m["alphabet"]) for ln in lines], given)
        smp = S.Sampler(Lattices(lat, m["ln_w"]))
        g = f"--given={TAPE[given]}"
        _cli([f"--decode={d}/k5", g, "-k", "5", sf, fst])
        _cli([f"--decode={d}/k5s", g, "-k", "5", f"--sum={d}/sum0", sf, fst])
        assert open(f"{d}/k5").read() == open(f"{d}/k5s").read()
        err = _cli([f"--decode={d}/smp", g, f"--sample={n}", "-R", "9", f"--sum={d}/sum", sf, fst])
        assert f"{n} derivations drawn per string (seed 9)" in err and "Sum: total weights of" in err, err
        assert open(f"{d}/sum").read() == open(f"{d}/sum0").read()
        sums = [float(x) for x in open(f"{d}/sum").read().split()]
        got = D.read_decode(f"{d}/smp", n)
        assert len(sums) == len(got) == len(lines)
        kept = {int(e): i for i, e in enumerate(lat["kept"])}
        exempt = 0
        for e in range(len(lines)):
            if e not in kept:
                assert sums[e] == -math.inf and all(x == (-math.inf, (), "") for x in got[e])
                continue
            exempt += _check_lattice(smp, kept[e], sums[e], [x[:2] for x in got[e]], 9, e)
            for w, p, s in got[e]:
                assert s == D.decoded_string(m, p, given)
        assert exempt <= 0.001 * n * len(kept)


@pytest.mark.parametrize("given", [0, 1])
@pytest.mark.parametrize("seed", range(2))
def test_free_sum_is_the_sum_over_free_strings(native_lib, oracle_bin, tmp_path, seed, given):
    """2-member random cascades: --decode --sum of a string x equals the log-sum over every free string y up to the
    lattice's longest path of --viterbi --sum of the pair"""
    rng = np.random.default_rng(20272101 + 10 * seed + given)
    d = str(tmp_path)
    a, b = os.path.join(d, "a.fst"), os.path.join(d, "b.fst")
    model = ["--train-cascade", a, b]
    for _ in range(50):
        _, ta = D.random_machine(rng, n_states=int(rng.integers(2, 4)), n_in=2, n_out=2, eps_rate=0.2, out_prefix="m")
        _, tb = D.random_machine(rng, n_states=int(rng.integers(2, 4)), n_in=2, n_out=2, eps_rate=0.2, in_prefix="m")
        open(a, "w").write(ta)
        open(b, "w").write(tb)
        open(os.path.join(d, "empty.data"), "w").close()
        if run(oracle_bin, ["--train-cascade", f"--dump-estimate={d}/e", os.path.join(d, "empty.data"), a, b])[0] == 0:
            break
    names = [f'"{"io"[given]}{j}"' for j in range(2)]
    lines = [" ".join(p) for k in range(3) for p in itertools.product(names, repeat=k)]
    sf = os.path.join(d, "s.txt")
    open(sf, "w").write("\n".join(lines) + "\n")
    _cli([f"--decode={d}/dec", f"--given={TAPE[given]}", f"--sum={d}/sum", sf, *model])
    sums = [float(x) for x in open(f"{d}/sum").read().split()]
    m = D.reference_model(oracle_bin, d, model)
    lat = D.free_lattices(m, [D.symbols(ln, m["alphabet"]) for ln in lines], given)
    free = m["arc_out"] if given == 0 else m["arc_in"]
    alphabet = sorted({m["names"][int(x)] for x in free if x})
    checked = 0
    for i, e in enumerate(lat["kept"]):
        bound = D.longest_path(lat, i)
        if len(alphabet) ** bound > 2000:
            continue
        xs = [" ".join(p) for k in range(bound + 1) for p in itertools.product(alphabet, repeat=k)]
        pairs = [(lines[e], x) if given == 0 else (x, lines[e]) for x in xs]
        open(f"{d}/pairs.data", "w").write("".join(f"{p}\n{q}\n" for p, q in pairs))
        _cli([f"--viterbi={d}/v", f"--sum={d}/psum", f"{d}/pairs.data", *model])
        ps = [float(x) for x in open(f"{d}/psum").read().split()]
        assert len(ps) == len(xs)
        fin = [x for x in ps if x > -math.inf]
        mx = max(fin)
        want = mx + math.log(math.fsum(math.exp(x - mx) for x in fin))
        assert _close(want, sums[e]), (e, want, sums[e])
        checked += 1
    assert checked >= 1


def _context(t, ln_w):
    from carmel_b200 import api as cb
    ctx = cb.Context(0, 64, cb.SPACE_LOG)
    for opt, v in ((cb.OPT_NO_ELL, 1), (cb.OPT_LANE_MIN, 0), (cb.OPT_NO_WIDE, 1)):
        ctx.set_option(opt, v)
    ctx.set_trivial_model(t["n_arcs_table"])
    ctx.set_params(ln_w)
    ctx.add_trellises(t["ex_states"], t["ex_fin"], t["ex_weight"], t["arc_off"], t["arc_dst"], t["arc_id"])
    return ctx


def test_distribution_on_random_lattices(native_lib):
    """20 random lattices, 100,000 draws each: the chi-square rule; sums and the first 2,000 draws under the reference"""
    rng = np.random.default_rng(20272201)
    t, ln_w = S.random_lattices(rng, 40, n_states=(4, 8), zero_rate=0.05)
    lat = Lattices(t, ln_w)
    smp = S.Sampler(lat)
    keys = np.arange(t["n_ex"], dtype=np.uint64) * 7919 + 11
    ctx = _context(t, ln_w)
    n = 100000
    tot, w, ln, b, a = ctx.sample(n, 3, keys)
    checked = 0
    for e in range(t["n_ex"]):
        got = [(float(w[e, r]), tuple(int(x) for x in a[b[e * n + r]:b[e * n + r] + ln[e, r]])) for r in range(n)]
        if smp.ln_total(e) == -math.inf or len(lat.paths(e)) < 3 or checked == 20:
            assert smp.ln_total(e) > -math.inf or tot[e] == -math.inf
            continue
        assert S.chi2_fit(lat, e, [p for _, p in got]) > 1e-6, e
        assert _check_lattice(smp, e, tot[e], got[:2000], 3, int(keys[e])) <= 2
        checked += 1
    assert checked == 20
    ctx.close()


def test_cli_epron_jpron_and_cipher(native_lib, tmp_path):
    """--sample / --sum on the trained epron-jpron (--decode) and the cipher (--viterbi): a string's sample lines do not
    change when another line becomes underivable, --sum leaves the decode files unchanged, read_kbest / read_decode parse
    the sample files"""
    d = str(tmp_path)
    data, fst = stage(tmp_path, "epron-jpron.data", "epron-jpron.fst")
    trained = os.path.join(d, "epron-jpron.fst.trained")
    _cli(["-t", "-F", trained, data, fst])
    jp = open(data).read().splitlines()[1::2]
    open(f"{d}/a.txt", "w").write("\n".join(jp) + "\n")
    open(f"{d}/b.txt", "w").write("\n".join(jp[:1] + ['"no-such-symbol"'] + jp[2:]) + "\n")
    n = 20
    for f in ("a", "b"):
        _cli([f"--decode={d}/{f}.smp", "--given=output", f"--sample={n}", f"--sum={d}/{f}.sum", f"{d}/{f}.txt", trained])
    sa, sb = open(f"{d}/a.smp").read().splitlines(), open(f"{d}/b.smp").read().splitlines()
    assert len(sa) == len(sb) == n * len(jp)
    assert sb[n:2 * n] == ["-inf 0 | ||"] * n
    assert sa[:n] == sb[:n] and sa[2 * n:] == sb[2 * n:]
    ua, ub = open(f"{d}/a.sum").read().split(), open(f"{d}/b.sum").read().split()
    assert ub[1] == "-inf" and ua[:1] + ua[2:] == ub[:1] + ub[2:] and float(ua[1]) > -math.inf
    assert len(D.read_decode(f"{d}/a.smp", n)) == len(jp)
    _cli([f"--decode={d}/v1", "--given=output", f"{d}/a.txt", trained])
    _cli([f"--decode={d}/v2", "--given=output", f"--sum={d}/x.sum", f"{d}/a.txt", trained])
    assert open(f"{d}/v1").read() == open(f"{d}/v2").read() and open(f"{d}/x.sum").read() == open(f"{d}/a.sum").read()
    # cipher pairs: the --viterbi / -k files are unchanged by --sum; the sample file parses as a -k file
    cdata, wfsa, cfst = stage(tmp_path, "cipher.data", "cipher.wfsa", "cipher.fst")
    open(cfst, "w").write(open(os.path.join(GOLDEN, "cipher.fst.trained")).read())
    args = ["--train-cascade", cdata, wfsa, cfst]
    for k in ([], ["-k", "5"]):
        _cli([f"--viterbi={d}/c1", *k, *args])
        _cli([f"--viterbi={d}/c2", *k, f"--sum={d}/c.sum", *args])
        assert open(f"{d}/c1").read() == open(f"{d}/c2").read()
    err = _cli([f"--viterbi={d}/cs", "--sample=7", f"--sum={d}/c2.sum", *args])
    assert "Sample: 7 derivations drawn per example (seed 1)" in err, err
    assert open(f"{d}/c.sum").read() == open(f"{d}/c2.sum").read()
    rows = read_kbest(f"{d}/cs", 7)
    assert len(rows) == 10 and all(w > -math.inf for ex in rows for w, _ in ex)
    _cli([f"--viterbi={d}/cs2", "--sample=7", "-R", "1", *args])
    assert open(f"{d}/cs").read() == open(f"{d}/cs2").read()


def _big_lattices(seed, n_ex, n_states):
    rng = np.random.default_rng(seed)
    return S.random_lattices(rng, n_ex, n_states=n_states, zero_rate=0.02)


def test_chunks_determinism_and_errors(native_lib, tmp_path):
    from carmel_b200 import api as cb
    t, ln_w = _big_lattices(20272301, 1200, (300, 500))
    assert int(t["ex_states"].sum()) * 8 > 3 << 20
    ctx = _context(t, ln_w)
    one = ctx.sample(6, 42)
    st = ctx.sample_stats()
    assert st["chunks"] == 1 and st["scratch_bytes"] == 8 * int(t["ex_states"].sum())
    again = ctx.sample(6, 42)
    ctx.set_option(cb.OPT_KBEST_SCRATCH_MB, 1)
    split = ctx.sample(6, 42)
    assert ctx.sample_stats()["chunks"] >= 3
    for other in (again, split):
        for x, y in zip(one, other):
            assert x.tobytes() == y.tobytes()
    smp = S.Sampler(Lattices(t, ln_w))
    tot, w, ln, b, a = one
    for e in range(0, t["n_ex"], 97):
        _check_lattice(smp, e, tot[e], _rows(w[e:e + 1], ln[e:e + 1], b[e * 6:], a)[0], 42, e)
    with pytest.raises(cb.CarmelB200Error) as ex:
        ctx.sample(3, 1, cap=5)
    assert ex.value.code == cb.ERR_ARG
    ctx.close()
    # an *e*:*e* loop puts a cycle into every lattice
    f, c = os.path.join(str(tmp_path), "c.fst"), os.path.join(str(tmp_path), "c.data")
    open(f, "w").write('qf\n(q0 (q0 "a" "x" 0.5))\n(q0 (q1 *e* *e* 0.3))\n(q1 (q0 *e* *e* 0.4))\n(q1 (qf "b" "z" 0.6))\n')
    open(c, "w").write('"a" "a" "b"\n"x" "x" "z"\n"a" "b"\n"x" "z"\n')
    job = cb.Job(["-t", "--no-ell", "--no-dense", "--no-lane", c, f])
    ctx = job.prepare()
    for n in (0, 3):
        with pytest.raises(cb.CarmelB200Error) as ex:
            ctx.sample(n, 1)
        assert ex.value.code == cb.ERR_CYCLE
    job.close()
