"""The CPU reference for sums and samples (sample_helpers.Sampler) against brute-force enumeration of every derivation,
its draws against the distribution they sample (chi-square rule of sample_helpers.py), and the --sample / --sum argument
handling of the command line.  CPU only."""
import math
import os

import numpy as np
import pytest

import sample_helpers as S
from helpers import random_wfst, read_estimate_dump, read_trellis_dump, run, sample_pairs, stage
from kbest_helpers import Lattices


def _brute_total(lat, e):
    ws = [w for w, _ in lat.paths(e) if w > -math.inf]
    if not ws:
        return -math.inf
    m = max(ws)
    return m + math.log(math.fsum(math.exp(w - m) for w in ws))


def test_uniform_restates_splitmix64():
    assert int(S.mix64(np.uint64(0))) == 0xE220A8397B1DCDAF  # splitmix64's first output from state 0
    u = S.sample_uniform(7, 3, np.arange(1000), 2)
    assert u.min() >= 0.0 and u.max() < 1.0 and len(set(u.tolist())) == 1000
    assert S.sample_uniform(7, 3, 5, 2) == u[5] and S.sample_uniform(7, 4, 5, 2) != u[5]


def test_total_is_the_sum_over_all_derivations(oracle_bin, tmp_path):
    rng = np.random.default_rng(20271701)
    t, ln_w = S.random_lattices(rng, 60, zero_rate=0.3)
    lats = [Lattices(t, ln_w)]
    for seed in range(3):  # and the oracle's pair lattices of random transducers
        r = np.random.default_rng(20271711 + seed)
        ns = int(r.integers(2, 6))
        fst, ins, outs, arcs = random_wfst(r, n_states=ns, eps_rate=float(r.uniform(0, 0.3)))
        d = str(tmp_path / f"s{seed}")
        os.makedirs(d)
        open(f"{d}/r.fst", "w").write(fst)
        open(f"{d}/r.data", "w").write(sample_pairs(r, arcs, ns, n_pairs=8, max_steps=6, ins=ins, outs=outs))
        rc, _, err = run(oracle_bin, ["-t", f"--dump-trellis={d}/t", f"--dump-estimate={d}/e", f"{d}/r.data", f"{d}/r.fst"])
        assert rc == 0, err
        lats.append(Lattices(read_trellis_dump(f"{d}/t"), read_estimate_dump(f"{d}/e")["ln_w"]))
    n_inf = 0
    for lat in lats:
        smp = S.Sampler(lat)
        for e in range(lat.t["n_ex"]):
            want, got = _brute_total(lat, e), smp.ln_total(e)
            if want == -math.inf:
                n_inf += 1
                assert got == -math.inf, (e, got)
                assert smp.draw(e, 1, e, 3)[0] == [(), (), ()]
            else:
                assert abs(got - want) <= 1e-12 * max(1.0, abs(want)), (e, got, want)
    assert n_inf >= 1  # some random lattice has no derivation of non-zero weight


@pytest.mark.parametrize("seed", [11, 12, 13])
def test_reference_draws_fit_the_distribution(seed):
    """200,000 draws of each of 4 random lattices against exp(ln w - ln total); every draw a derivation of its weight"""
    rng = np.random.default_rng(20271800 + seed)
    t, ln_w = S.random_lattices(rng, 12, n_states=(4, 8), zero_rate=0.05)
    lat = Lattices(t, ln_w)
    smp = S.Sampler(lat)
    done = 0
    for e in range(t["n_ex"]):
        if smp.ln_total(e) == -math.inf or len(lat.paths(e)) < 3 or done == 4:
            continue
        paths, w, exempt = smp.draw(e, seed, 1000 + e, 200000)
        assert S.chi2_fit(lat, e, paths) > 1e-6, e
        for p, x in list(zip(paths, w))[:2000]:
            assert lat.weight(e, p) == x, (p, x)
        assert (exempt >= 0).sum() <= 200  # 0.1 %
        done += 1
    assert done == 4


def _cli(args):
    from carmel_b200 import CLI_PATH
    return run(CLI_PATH, args)


@pytest.mark.parametrize("bad", [["--sample=2", "-k", "3"], ["--sample=2", "-k", "1"], ["--sample=0"], ["--sample="],
                                 ["--sample"], ["--sample=x"], ["--sample=-1"], ["--sample=2x"], ["--sample=4294967296"],
                                 ["--sum="], ["--sum"]])
def test_refusals(native_lib, tmp_path, bad):
    data, fst = stage(tmp_path, "epron-jpron.data", "epron-jpron.fst")
    strings = os.path.join(str(tmp_path), "s.txt")
    open(strings, "w").write("".join(open(data).readlines()[1::2]))
    for mode in ([f"--viterbi={tmp_path}/v", "-t", data], [f"--decode={tmp_path}/d", "--given=output", strings]):
        rc, _, err = _cli([mode[0], *bad, *mode[1:], fst])
        assert rc == -9 % 256, (mode, bad, rc, err)
        assert "--sample" in err or "--sum" in err, err
        assert not os.path.exists(f"{tmp_path}/v") and not os.path.exists(f"{tmp_path}/d")


def test_options_without_a_decode_are_unused(native_lib, tmp_path):
    """without --viterbi / --decode, --sample and --sum are unknown long options, accepted and unused, as -k is: the run
    exits and writes as it does without them"""
    data, fst = stage(tmp_path, "epron-jpron.data", "epron-jpron.fst")
    base = _cli(["-t", "-M", "2", data, fst])
    for extra in (["--sample=0", "--sum="], ["--sample=3", "-k", "2", f"--sum={tmp_path}/s"], ["--sample=x"]):
        got = _cli(["-t", "-M", "2", *extra, data, fst])
        assert got[0] == base[0] and got[1] == base[1], (extra, got[0], base[0], got[2])
        assert not os.path.exists(f"{tmp_path}/s")
