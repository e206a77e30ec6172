"""k-best decode on the GPU (cml_kbest / k_kbest, carmel-b200 --viterbi=FILE -k n) against the CPU reference (a lazy
enumeration over the oracle's lattices, kbest_helpers.Lattices.kbest) under the comparison rule of kbest_helpers.py, the
rank-0 line against the 1-best decode, and the C ABI's chunking, determinism and errors."""
import math
import os

import numpy as np
import pytest

from helpers import GOLDEN, random_wfst, read_estimate_dump, read_trellis_dump, run, sample_pairs, stage
from kbest_helpers import Lattices, compare_kbest, read_kbest

pytestmark = pytest.mark.gpu


def _lattices(oracle_bin, d, args):
    rc, _, err = run(oracle_bin, [f"--dump-trellis={d}/t", f"--dump-estimate={d}/e", *args], timeout=600)
    assert rc == 0, err
    return Lattices(read_trellis_dump(f"{d}/t"), read_estimate_dump(f"{d}/e")["ln_w"])


def _decode_both(lat, d, args, k):
    """(reference lists, GPU lists, GPU log); checks that every example's rank-0 line is its --viterbi (k = 1) line"""
    from carmel_b200 import CLI_PATH
    rc, _, err = run(CLI_PATH, [f"--viterbi={d}/v.p", "-k", str(k), *args], timeout=600)
    assert rc == 0, err
    rc, _, err1 = run(CLI_PATH, [f"--viterbi={d}/v1.p", *args], timeout=600)
    assert rc == 0, err1
    lines_k, lines_1 = open(f"{d}/v.p").read().splitlines(), open(f"{d}/v1.p").read().splitlines()
    assert len(lines_k) == k * len(lines_1)
    for e, ln in enumerate(lines_1):  # rank 0 is the 1-best decode, byte for byte
        assert lines_k[e * k] == ln, (e, lines_k[e * k], ln)
    return [lat.kbest(e, k) for e in range(lat.t["n_ex"])], read_kbest(f"{d}/v.p", k), err


def _check(want, got, lat):
    assert len(want) == len(got)
    for e, (w, g) in enumerate(zip(want, got)):
        compare_kbest(w, g, lambda p, e=e: lat.weight(e, p))
        for gw, gp in g:  # every listed path is a real derivation of the stated weight
            if gw > -math.inf:
                pw = lat.weight(e, gp)
                assert pw is not None and abs(pw - gw) <= 1e-9 * max(1.0, abs(gw)), (e, gp, pw, gw)


@pytest.mark.parametrize("seed", range(6))
def test_kbest_random_transducers(native_lib, oracle_bin, tmp_path, seed):
    rng = np.random.default_rng(20271101 + seed)
    ns = int(rng.integers(2, 7))
    fst, ins, outs, arcs = random_wfst(rng, n_states=ns, eps_rate=float(rng.uniform(0, 0.4)))
    corpus = sample_pairs(rng, arcs, ns, n_pairs=12, max_steps=7, ins=ins, outs=outs)
    d = str(tmp_path)
    f, c = os.path.join(d, "r.fst"), os.path.join(d, "r.data")
    open(f, "w").write(fst)
    open(c, "w").write(corpus)
    lat = _lattices(oracle_bin, d, ["-t", c, f])
    every = [sorted((w for w, _ in lat.paths(e) if w > -math.inf), reverse=True) for e in range(lat.t["n_ex"])]
    for k in (4, max(len(x) for x in every) + 3):
        want, got, _ = _decode_both(lat, d, ["-t", c, f], k)
        _check(want, got, lat)
        for e, ws in enumerate(every):  # brute force: the weights are the top k of all derivations
            top = (ws + [-math.inf] * k)[:k]
            for r, (tw, (gw, _)) in enumerate(zip(top, got[e])):
                assert tw == gw == -math.inf or abs(tw - gw) <= 1e-9 * max(1.0, abs(tw)), (e, r, tw, gw)


@pytest.mark.parametrize("trained", [True, False])
def test_kbest_cipher(native_lib, oracle_bin, tmp_path, trained):
    """the tutorial's decode: cipher.wfsa o cipher.fst(.trained), k = 5.  The untrained channel's uniform weights make
    exact ties, so the rank-0 line equal to the 1-best line also pins the tie key."""
    data, wfsa = stage(tmp_path, "cipher.data", "cipher.wfsa")
    fst = os.path.join(str(tmp_path), "cipher.fst")
    open(fst, "w").write(open(os.path.join(GOLDEN, "cipher.fst.trained" if trained else "cipher.fst")).read())
    args = ["--train-cascade", data, wfsa, fst]
    lat = _lattices(oracle_bin, str(tmp_path), args)
    want, got, err = _decode_both(lat, str(tmp_path), args, 5)
    assert "Viterbi: best derivations of 10 examples" in err
    assert "Viterbi: 5-best lists, 50 derivations found" in err
    _check(want, got, lat)


def test_kbest_tagging(native_lib, oracle_bin, tmp_path):
    """the first 20 tagging.data sentences through tagging.fsa o tagging.fst, k = 10"""
    src, fsa, fst = stage(tmp_path, "tagging.data", "tagging.fsa", "tagging.fst")
    data = os.path.join(str(tmp_path), "t20.data")
    open(data, "w").write("".join(open(src).readlines()[:40]))
    args = ["--train-cascade", data, fsa, fst]
    lat = _lattices(oracle_bin, str(tmp_path), args)
    want, got, _ = _decode_both(lat, str(tmp_path), args, 10)
    assert len(got) == 20
    _check(want, got, lat)


def test_bundled_k_binds_first(native_lib, tmp_path):
    """-Mk 7 3: carmel's priority chain binds k before M, so the file has 7 lines per example"""
    from carmel_b200 import CLI_PATH
    data, wfsa, fst = stage(tmp_path, "cipher.data", "cipher.wfsa", "cipher.fst")
    rc, _, err = run(CLI_PATH, ["--train-cascade", f"--viterbi={tmp_path}/v", "-Mk", "7", "3", data, wfsa, fst])
    assert rc == 0, err
    assert len(open(f"{tmp_path}/v").readlines()) == 70


def _cipher_job(tmp_path, extra=()):
    from carmel_b200 import Job
    data, wfsa, fst = stage(tmp_path, "cipher.data", "cipher.wfsa", "cipher.fst")
    open(fst, "w").write(open(os.path.join(GOLDEN, "cipher.fst.trained")).read())
    job = Job(["--train-cascade", "--no-ell", "--no-dense", "--no-lane", *extra, data, wfsa, fst])
    return job, job.prepare()


def test_kbest_chunks_and_determinism(native_lib, tmp_path):
    from carmel_b200 import api as cb
    job, ctx = _cipher_job(tmp_path)
    k = 40
    one = ctx.kbest(k)
    st = ctx.kbest_stats()
    assert st["chunks"] == 1 and st["scratch_bytes"] > 0
    again = ctx.kbest(k)
    ctx.set_option(cb.OPT_KBEST_SCRATCH_MB, 1)
    split = ctx.kbest(k)
    assert ctx.kbest_stats()["chunks"] > 1
    for a in (again, split):
        for x, y in zip(one, a):
            assert x.tobytes() == y.tobytes()
    w1, l1, b1, a1 = ctx.viterbi()
    w, ln, b, a = one
    assert w1[:, 0].tobytes() == w[:, 0].tobytes() and l1[:, 0].tobytes() == ln[:, 0].tobytes()
    for e in range(w.shape[0]):
        assert a1[b1[e]:b1[e] + l1[e, 0]].tolist() == a[b[e * k]:b[e * k] + ln[e, 0]].tolist()
        assert all(w[e, r] >= w[e, r + 1] for r in range(k - 1))
    job.close()


def test_kbest_errors(native_lib, tmp_path):
    from carmel_b200 import api as cb
    job, ctx = _cipher_job(tmp_path)
    for k, cap, code in ((0, None, cb.ERR_ARG), (3, 5, cb.ERR_ARG)):
        with pytest.raises(cb.CarmelB200Error) as ex:
            ctx.kbest(k, cap)
        assert ex.value.code == code
    job.close()
    os.makedirs(tmp_path / "s")
    job, ctx = _cipher_job(tmp_path / "s", ["--scaled"])
    with pytest.raises(cb.CarmelB200Error) as ex:
        ctx.kbest(3)
    assert ex.value.code == cb.ERR_STATE
    job.close()
    # an *e*:*e* loop puts a cycle into every lattice
    f, c = os.path.join(str(tmp_path), "c.fst"), os.path.join(str(tmp_path), "c.data")
    open(f, "w").write('qf\n(q0 (q0 "a" "x" 0.5))\n(q0 (q1 *e* *e* 0.3))\n(q1 (q0 *e* *e* 0.4))\n(q1 (qf "b" "z" 0.6))\n')
    open(c, "w").write('"a" "a" "b"\n"x" "x" "z"\n"a" "b"\n"x" "z"\n')
    job = cb.Job(["-t", "--no-ell", "--no-dense", "--no-lane", c, f])
    ctx = job.prepare()
    with pytest.raises(cb.CarmelB200Error) as ex:
        ctx.kbest(3)
    assert ex.value.code == cb.ERR_CYCLE
    job.close()
