"""Sums and samples of derivation lattices (cml_sample, carmel-b200 --sum / --sample): the CPU reference the parity tests
and bench_sample.py hold the GPU to, and the chi-square rule the distribution tests apply.

The reference works on the lattices kbest_helpers.Lattices holds (the oracle's --dump-trellis / --dump-estimate for
pairs, decode_helpers.free_lattices for free strings: the reference's state ids and stored arc order).  It takes beta by
memoised recursion from the start state instead of the GPU's level-by-level pass, restates sample_uniform of
include/carmel_b200.h in numpy uint64 arithmetic, and walks every draw of a lattice at once.  For every draw it records
the decision margin of each step: the smallest |c| after a subtraction up to the chosen arc.  Where that margin is below
1e-9, last-bit differences between two correct implementations (exp, the order of the log-sum-exp) can change the
choice, so a comparison is exempt from that step on.

Comparison rule (draws): sample r of lattice e equals the reference's arc for arc, up to its first step with margin
< 1e-9 (the sample is then exempt from that step on); exempt samples are at most 0.1 % of the samples.

Chi-square rule (distribution): the draws of a lattice are counted per path; the expected count of a path is
N * exp(ln w - ln total) from enumeration; cells of expected count < 5 are pooled into one; a drawn path that is not a
derivation of non-zero weight fails; the fit passes at p > 1e-6.
"""
import math
import sys

import numpy as np

from kbest_helpers import Lattices

MARGIN = 1e-9
_C0, _C1, _C2 = np.uint64(0x9E3779B97F4A7C15), np.uint64(0xBF58476D1CE4E5B9), np.uint64(0x94D049BB133111EB)


def mix64(x):
    """splitmix64 finaliser on uint64 arrays (wrapping arithmetic)"""
    x = np.asarray(x, np.uint64)
    with np.errstate(over="ignore"):
        x = x + _C0
        x = (x ^ (x >> np.uint64(30))) * _C1
        x = (x ^ (x >> np.uint64(27))) * _C2
    return x ^ (x >> np.uint64(31))


def sample_uniform(seed, key, r, t):
    """u of sample(s) r (int or array) at step t: h = mix64(seed ^ mix64(key)); h = mix64(h + (r << 32 | t));
    u = (h >> 11) * 2^-53"""
    h0 = mix64(np.uint64(seed) ^ mix64(np.uint64(key)))
    ctr = (np.asarray(r, np.uint64) << np.uint64(32)) | np.uint64(t)
    with np.errstate(over="ignore"):
        h = mix64(h0 + ctr)
    return (h >> np.uint64(11)).astype(np.float64) * 2.0 ** -53


def _lse(v):
    m = max(v, default=-math.inf)
    if m == -math.inf:
        return -math.inf
    return m + math.log(sum(math.exp(x - m) for x in v))


class Sampler:
    """beta, ln total and draws of the lattices of a kbest_helpers.Lattices"""

    def __init__(self, lat: Lattices):
        self.L = lat
        self._beta = {}

    def _arcs(self, e, s):
        off, dst, aid = self.L.rows[e], self.L.t["arc_dst"], self.L.t["arc_id"]
        return [(int(dst[k]), int(aid[k]), float(self.L.ln_w[aid[k]])) for k in range(off[s], off[s + 1])]

    def beta(self, e):
        """[ln sum over paths s -> goal of their weight] per state of lattice e (memoised recursion from the start)"""
        if e in self._beta:
            return self._beta[e]
        n, fin = len(self.L.rows[e]) - 1, int(self.L.t["ex_fin"][e])
        b = [None] * n
        sys.setrecursionlimit(max(sys.getrecursionlimit(), 4 * n + 1000))

        def get(s):
            if b[s] is None:
                b[s] = 0.0 if s == fin else _lse([w + get(d) for d, _, w in self._arcs(e, s)])
            return b[s]

        for s in range(n):
            get(s)
        self._beta[e] = b
        return b

    def ln_total(self, e):
        return self.beta(e)[0]

    def draw(self, e, seed, key, n):
        """n draws of lattice e: (paths [tuple of arc ids] * n, ln weights [n], exempt [n]: index of the first step with
        margin < 1e-9, or -1)"""
        b, fin = self.beta(e), int(self.L.t["ex_fin"][e])
        if b[0] == -math.inf:
            return [()] * n, np.full(n, -math.inf), np.full(n, -1)
        cur = np.zeros(n, np.int64)
        w = np.zeros(n)
        exempt = np.full(n, -1)
        ids = np.full((n, len(b)), -1, np.int64)  # a path visits each state at most once
        t = 0
        while True:
            act = np.nonzero(cur != fin)[0]
            if act.size == 0:
                break
            u = sample_uniform(seed, key, act, t)
            src = cur[act]
            for s in np.unique(src):
                sel = src == s
                idx, c = act[sel], u[sel].copy()
                arcs = self._arcs(e, int(s))
                ps = [math.exp(lw + b[d] - b[s]) for d, _, lw in arcs]
                chosen = np.full(idx.size, -1)
                margin = np.full(idx.size, math.inf)
                for j, p in enumerate(ps):
                    if p > 0:
                        und = chosen < 0
                        c[und] -= p
                        margin[und] = np.minimum(margin[und], np.abs(c[und]))
                        chosen[und & (c < 0)] = j
                chosen[chosen < 0] = max(j for j, p in enumerate(ps) if p > 0)  # rounding: the last arc with p > 0
                exempt[idx[(exempt[idx] < 0) & (margin < MARGIN)]] = t
                dst, aid, lws = (np.array([a[k] for a in arcs]) for k in range(3))
                cur[idx] = dst[chosen]
                w[idx] += lws[chosen]
                ids[idx, t] = aid[chosen]
            t += 1
        paths = [tuple(int(x) for x in row[row >= 0]) for row in ids]
        return paths, w, exempt


def compare_draws(want, got):
    """the comparison rule on one lattice: want = Sampler.draw's (paths, weights, exempt), got = [(ln w, arc ids)] * n.
    Returns the number of exempt samples."""
    wp, ww, ex = want
    assert len(wp) == len(got)
    n_ex = 0
    for r, ((gw, gp), p) in enumerate(zip(got, wp)):
        if ex[r] >= 0:
            n_ex += 1
            assert tuple(gp[:ex[r]]) == p[:ex[r]], (r, gp, p, ex[r])
            continue
        assert tuple(gp) == p, (r, gp, p)
        assert gw == ww[r] or abs(gw - ww[r]) <= 1e-12 * max(1.0, abs(gw)), (r, gw, ww[r])
    return n_ex


def chi2_fit(lat: Lattices, e, paths):
    """the chi-square rule: p value of the drawn paths of lattice e against enumeration"""
    from scipy.stats import chi2
    every = [(w, p) for w, p in lat.paths(e) if w > -math.inf]
    tot = _lse([w for w, _ in every])
    prob = {p: math.exp(w - tot) for w, p in every}
    count = {}
    for p in paths:
        assert p in prob, ("not a derivation of non-zero weight", p)
        count[p] = count.get(p, 0) + 1
    N = len(paths)
    big = [(N * q, count.get(p, 0)) for p, q in prob.items() if N * q >= 5]
    pool_e = sum(N * q for q in prob.values() if N * q < 5)
    pool_o = sum(count.get(p, 0) for p, q in prob.items() if N * q < 5)
    cells = big + ([(pool_e, pool_o)] if pool_e > 0 else [])
    if len(cells) < 2:
        return 1.0
    stat = sum((o - x) ** 2 / x for x, o in cells)
    return float(chi2.sf(stat, len(cells) - 1))


def random_lattices(rng, n_ex, n_states=(3, 9), zero_rate=0.1):
    """a batch in the --dump-trellis dict shape and ln weights per arc id (arc ids = global arc numbers, so a path is
    its id sequence): states 0..n-1 in topological order, the goal n-1; every state is reached from the start and
    reaches the goal; some arcs have weight zero (ln -inf), which can leave states, or a whole lattice, without a
    derivation of non-zero weight; parallel arcs occur"""
    ex_states, ex_fin, arc_off, arc_dst, arc_id, ln_w = [], [], [], [], [], []
    for _ in range(n_ex):
        n = int(rng.integers(n_states[0], n_states[1] + 1))
        out = [[] for _ in range(n)]
        for d in range(1, n):  # an in-arc from an earlier state
            out[int(rng.integers(0, d))].append(d)
        for s in range(n - 1):
            if not out[s]:
                out[s].append(int(rng.integers(s + 1, n)))
            for _ in range(int(rng.integers(0, 3))):
                out[s].append(int(rng.integers(s + 1, n)))
            rng.shuffle(out[s])
        off = [0]
        for s in range(n):
            for d in out[s]:
                arc_dst.append(d)
                arc_id.append(len(ln_w))
                ln_w.append(-math.inf if rng.random() < zero_rate else float(np.log(rng.uniform(0.02, 1.0))))
            off.append(off[-1] + len(out[s]))
        ex_states.append(n)
        ex_fin.append(n - 1)
        arc_off.append(np.asarray(off, np.uint32))
    u32 = lambda x: np.asarray(x, np.uint32)
    t = dict(n_ex=n_ex, n_arcs_table=len(ln_w), ex_states=u32(ex_states), ex_fin=u32(ex_fin),
             ex_weight=np.ones(n_ex), arc_off=np.concatenate(arc_off).astype(np.uint32), arc_dst=u32(arc_dst),
             arc_id=u32(arc_id))
    return t, np.asarray(ln_w, np.float64)
