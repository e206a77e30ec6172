"""The CPU reference for decoding strings with the other tape free (decode_helpers.free_lattices: memoised recursion over
(state, position), then a sort into the numbering of include/carmel_b200.h) against brute-force enumeration of every
accepting machine path whose given tape spells the string, and the --decode argument handling of the command line.
CPU only."""
import os

import numpy as np
import pytest

from decode_helpers import GivenEpsCycle, eps_levels, free_lattices, random_machine
from helpers import run, stage
from kbest_helpers import Lattices


def _brute_force(m, s, given, ln_w):
    """{arc ids: ln weight} of every accepting machine path whose tape-`given` labels spell s"""
    glab = m["arc_in"] if given == 0 else m["arc_out"]
    off, dst, fin = m["state_arc_off"], m["arc_dest"], int(m["final_state"])
    bound = len(s) + (len(s) + 1) * (max(eps_levels(m, given)) + 1)  # a path's given-*e* arcs climb the eps-levels
    out, stack = {}, [(0, 0, (), 0.0)]
    while stack:
        q, t, ids, w = stack.pop()
        if q == fin and t == len(s):
            out[ids] = w
        assert len(ids) <= bound
        for a in range(off[q], off[q + 1]):
            if glab[a] == 0:
                stack.append((int(dst[a]), t, ids + (a,), w + ln_w[a]))
            elif t < len(s) and glab[a] == s[t]:
                stack.append((int(dst[a]), t + 1, ids + (a,), w + ln_w[a]))
    return out


@pytest.mark.parametrize("given", [0, 1])
@pytest.mark.parametrize("seed", range(6))
def test_reference_lattice_paths_are_the_machine_paths(seed, given):
    rng = np.random.default_rng(20271201 + seed)
    m, _ = random_machine(rng, n_states=int(rng.integers(2, 6)), eps_rate=float(rng.uniform(0.1, 0.4)))
    ln_w = np.log(rng.uniform(0.05, 1.0, m["arc_in"].size))
    lo, hi = (1, 4) if given == 0 else (4, 7)  # ids of the given tape's symbols
    strings = [[], [int(x) for x in rng.integers(lo, hi, 1)], [int(x) for x in rng.integers(lo, hi, 2)],
               [int(x) for x in rng.integers(lo, hi, 3)], [int(x) for x in rng.integers(lo, hi, 4)],
               [lo, 99], [0]]  # 99: a symbol no arc carries; 0 (*e*) matches no arc
    lat = free_lattices(m, strings, given)
    L = Lattices(lat, ln_w)
    assert sorted(lat["kept"].tolist() + lat["dropped"].tolist()) == list(range(len(strings)))
    assert 5 in lat["dropped"] and 6 in lat["dropped"]
    for i, e in enumerate(lat["kept"]):
        want = _brute_force(m, strings[e], given, ln_w)
        got = {ids: w for w, ids in L.paths(i)}
        assert set(got) == set(want), (e, strings[e])
        for ids, w in want.items():
            assert abs(got[ids] - w) <= 1e-12 * max(1.0, abs(w))
        # numbering: start = 0, goal = last, every arc goes to a later state
        n = int(lat["ex_states"][i])
        assert int(lat["ex_fin"][i]) == n - 1
        rows = L.rows[i]
        assert all(int(lat["arc_dst"][k]) > s for s in range(n) for k in range(rows[s], rows[s + 1]))
    for e in lat["dropped"]:
        assert not _brute_force(m, strings[e], given, ln_w), strings[e]


def test_reference_refuses_a_given_eps_cycle():
    m = dict(n_states=2, final_state=1, state_arc_off=np.array([0, 2, 3], np.uint32), arc_in=np.array([1, 0, 1], np.uint32),
             arc_out=np.array([0, 2, 0], np.uint32), arc_dest=np.array([1, 1, 0], np.uint32))
    assert free_lattices(m, [[1]], 0)["n_ex"] == 1  # input tape: no cycle of input-*e* arcs
    with pytest.raises(GivenEpsCycle):
        free_lattices(m, [[1]], 1)  # output tape: 0 -> 1 -> 0 has *e* outputs only


def test_decode_argument_refusals(native_lib, tmp_path):
    """--given missing or not input/output, --decode with --viterbi, --crp or a training switch, and a bad -k are refused
    with the argument-error exit before any work; nothing is written"""
    from carmel_b200 import CLI_PATH
    (fst,) = stage(tmp_path, "epron-jpron.fst")
    strings = os.path.join(str(tmp_path), "s.txt")
    open(strings, "w").write('"R" "I" "N"\n')
    out = os.path.join(str(tmp_path), "out")
    cases = [([], "--decode needs --given"), (["--given=both"], "--decode needs --given"),
             (["--given=output", f"--viterbi={out}.v"], "cannot be combined"),
             (["--given=output", "--crp"], "cannot be combined")]
    cases += [(["--given=output", "-k", bad], "-k needs") for bad in ("0", "x", "-2", "")]
    # switches that train or write what only training writes are refused rather than ignored
    cases += [(["--given=output", *flags], "cannot be combined with") for flags in
              (["-t"], ["-F", out + ".F"], ["-M", "3"], ["--trellis-only"], [f"--dump-trellis={out}.t"],
               [f"--history={out}.h"], [f"--fem-param={out}.p"])]
    for extra, msg in cases:
        rc, _, err = run(CLI_PATH, [f"--decode={out}", *extra, strings, fst])
        assert rc == -9 % 256 and msg in err, (extra, rc, err)
        assert not any(os.path.exists(out + x) for x in ("", ".v", ".F", ".t", ".h", ".p"))
    rc, _, err = run(CLI_PATH, [f"--decode={out}", "--given=output", "--gpus=2", strings, fst])
    assert rc == -11 % 256 and "--decode decodes on one GPU" in err, err
    assert not os.path.exists(out)


def test_decode_without_gpu_fails_loudly(native_lib, tmp_path):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    from carmel_b200 import CLI_PATH
    (fst,) = stage(tmp_path, "epron-jpron.fst")
    strings = os.path.join(str(tmp_path), "s.txt")
    open(strings, "w").write('"R" "I" "N"\n')
    rc, _, err = run(CLI_PATH, [f"--decode={tmp_path}/out", "--given=output", strings, fst])
    assert rc != 0 and ("no CPU fallback" in err or "CUDA" in err), err
    assert not (tmp_path / "out").exists()
