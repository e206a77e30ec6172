"""Sums and samples of derivation forests (cml_forests_sample, forest-em-b200 -v FILE --sample=n): the CPU reference the
parity tests and bench_forest_sample.py hold the GPU to, the comparison rule, enumeration and the chi-square rule.

The reference (ForestSampler) works on the pre-order arrays the library gets (forest_kbest_helpers.forests_to_arrays)
and uses a different algorithm from the GPU: inside values by memoised recursion from the root instead of a pass by
height, the uniforms of sample_helpers.sample_uniform (numpy uint64), and a recursive pre-order walk per sample.  For
every OR decision it records the margin: the distance of c from the nearest cumulative boundary, i.e. the smallest |c|
after a subtraction up to the chosen child.  Where that margin is below 1e-9, last-bit differences between two correct
implementations (exp, log) can change the choice, so a comparison is exempt from that decision on.

Comparison rule, per forest:
  * ln_total and every sample's ln weight agree to 1e-12 * max(1, |x|); -inf on both sides where there is none;
  * sample r's node sequence is identical to the reference's, up to the sample's first decision with a margin below
    1e-9 (the nodes recorded before that decision must agree; the rest of the sample is exempt);
  * at most 0.1 % of the samples may be exempted that way (checked over a whole comparison by the caller).

Chi-square rule (distribution): the draws of a forest are counted per node sequence; the expected count of a sequence
is N * (its probability from enumeration); cells of expected count < 5 are pooled into one; a drawn sequence that is
not a derivation of non-zero weight fails; the fit passes at p > 1e-6.
"""
import math
import sys

import numpy as np

from sample_helpers import sample_uniform

MARGIN = 1e-9
EXEMPT_SHARE = 1e-3


def _lse(v):
    m = max(v, default=-math.inf)
    if m == -math.inf:
        return -math.inf
    return m + math.log(sum(math.exp(x - m) for x in v))


class ForestSampler:
    """one forest's pre-order arrays and the rule weights (ln): inside values, ln total and draws"""

    def __init__(self, nxt, label, backref, ln_w):
        self.nx, self.lb, self.br = [int(x) for x in nxt], [int(x) for x in label], [int(x) for x in backref]
        self.ln_w = [float(x) for x in np.asarray(ln_w, np.float64)]
        n = len(self.nx)
        self.slots = [[] for _ in range(n)]  # real node -> its child slots, resolved to real nodes
        for p in range(n):
            if not self.br[p]:
                q = p + 1
                while q < self.nx[p]:
                    self.slots[p].append(self.lb[q] if self.br[q] else q)
                    q = self.nx[q]
        self.ins = [None] * n
        sys.setrecursionlimit(max(sys.getrecursionlimit(), 20 * n + 1000))

    def inside(self, v):
        """inside value of real node v: AND = ln_w[rule] + slots in order, OR = max-shifted log-sum-exp"""
        if self.ins[v] is None:
            if self.lb[v]:
                s = self.ln_w[self.lb[v]]
                for c in self.slots[v]:
                    s = s + self.inside(c)
                self.ins[v] = s
            else:
                self.ins[v] = _lse([self.inside(c) for c in self.slots[v]])
        return self.ins[v]

    def ln_total(self):
        return self.inside(0)

    def draw(self, seed, key, n):
        """n draws: (node sequences [tuple] * n, ln weights [n], exempt [n]: the number of leading nodes that must
        agree when the sample has a decision with margin < 1e-9, or -1)"""
        total = self.ln_total()
        if total == -math.inf:
            return [()] * n, np.full(n, -math.inf), np.full(n, -1)
        cols = {}

        def u_of(r, t):
            if t not in cols:
                cols[t] = sample_uniform(seed, key, np.arange(n), t)
            return float(cols[t][r])

        paths, weights, exempt = [], np.zeros(n), np.full(n, -1)
        for r in range(n):
            out, st = [], {"t": 0, "w": 0.0, "ex": -1}

            def visit(c):
                while not self.lb[c]:
                    x = u_of(r, st["t"])
                    st["t"] += 1
                    ic = self.inside(c)
                    pick, last, margin = None, None, math.inf
                    for d in self.slots[c]:
                        p = math.exp(self.inside(d) - ic)
                        if p > 0:
                            last = d
                            x -= p
                            margin = min(margin, abs(x))
                            if x < 0:
                                pick = d
                                break
                    if margin < MARGIN and st["ex"] < 0:
                        st["ex"] = len(out)
                    c = pick if pick is not None else last
                out.append(c)
                st["w"] += self.ln_w[self.lb[c]]
                for d in self.slots[c]:
                    visit(d)

            visit(0)
            paths.append(tuple(out))
            weights[r] = st["w"]
            exempt[r] = st["ex"]
        return paths, weights, exempt

    def derivations(self):
        """every derivation of non-zero weight as {node sequence: ln weight}, by enumeration (sequences from distinct
        choice sets that coincide are merged)"""
        memo = {}

        def rec(v):
            if v not in memo:
                if self.lb[v]:
                    out = [(self.ln_w[self.lb[v]], (v,))]
                    for c in self.slots[v]:
                        out = [(w + x, s + t) for w, s in out for x, t in rec(c)]
                else:
                    out = [d for c in self.slots[v] for d in rec(c)]
                memo[v] = [(w, s) for w, s in out if w > -math.inf]
            return memo[v]

        got = {}
        for w, s in rec(0):
            got.setdefault(s, []).append(w)
        return {s: _lse(ws) for s, ws in got.items()}


def forest_samplers(node_off, nxt, label, backref, ln_w):
    return [ForestSampler(nxt[int(node_off[i]):int(node_off[i + 1])], label[int(node_off[i]):int(node_off[i + 1])],
                          backref[int(node_off[i]):int(node_off[i + 1])], ln_w) for i in range(len(node_off) - 1)]


def _close(a, b):
    return a == b or abs(a - b) <= 1e-12 * max(1.0, abs(a))


def compare_samples(sampler, want, got_total, got):
    """the comparison rule on one forest: want = ForestSampler.draw's (paths, weights, exempt), got = [(ln w, node
    sequence)] * n.  Returns the number of exempt samples."""
    wt = sampler.ln_total()
    assert _close(wt, got_total), (wt, got_total)
    wp, ww, ex = want
    assert len(wp) == len(got)
    n_ex = 0
    for r, ((gw, gp), p) in enumerate(zip(got, wp)):
        if ex[r] >= 0:
            n_ex += 1
            assert tuple(gp[:ex[r]]) == p[:ex[r]], (r, gp, p, ex[r])
            continue
        assert tuple(gp) == p, (r, gp, p)
        assert _close(ww[r], gw), (r, gw, ww[r])
    return n_ex


def chi2_fit(sampler, paths):
    """the chi-square rule: p value of the drawn node sequences of one forest against enumeration"""
    from scipy.stats import chi2
    every = sampler.derivations()
    tot = _lse(list(every.values()))
    prob = {s: math.exp(w - tot) for s, w in every.items()}
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


def small_forests(rng, n_forests, n_rules, max_derivations=40):
    """random forests (forest_helpers.random_forest, shared nodes on) with at most max_derivations derivations each, so
    they can be enumerated and fitted"""
    from forest_helpers import random_forest
    from forest_kbest_helpers import forests_to_arrays
    texts = []
    while len(texts) < n_forests:
        t = random_forest(rng, n_rules, depth=int(rng.integers(1, 4)), share=0.25)
        _, nx, lb, br = forests_to_arrays([t])
        if 2 <= count_derivations(ForestSampler(nx, lb, br, np.zeros(n_rules + 1))) <= max_derivations:
            texts.append(t)
    return texts


def count_derivations(s):
    """number of derivations (choice sets, zero weights included) without enumerating them"""
    memo = {}

    def rec(v):
        if v not in memo:
            memo[v] = math.prod(rec(c) for c in s.slots[v]) if s.lb[v] else sum(rec(c) for c in s.slots[v])
        return memo[v]
    return rec(0)
