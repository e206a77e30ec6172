"""k-best derivations of derivation forests (forest-em-b200 -v FILE --kbest=n, cml_forests_kbest): the forests in the
library's pre-order arrays, the CPU reference the parity tests and bench_kbest.py hold the GPU to, the file reader and
the comparison rule.

The reference (ForestRef.kbest) works on the same pre-order arrays the library gets and uses a different algorithm
from the GPU: a lazy enumeration with a candidate heap per node (Huang & Chiang 2005, "Better k-best parsing",
algorithm 3), memoised per node, so a shared node (back reference) is computed once and used independently at every
use, instead of an eager k-best merge by height.

A derivation is written as the in-forest pre-order indices of its AND nodes, in derivation pre-order.

Comparison rule, rank by rank over the n derivations of a forest (the one of kbest_helpers.py, restated for trees):
  * scores agree within 1e-9 * max(1, |s|); padding (-inf) on both sides;
  * ranks are grouped into runs of equal score (within 1e-12 relative);
  * every run that ends before rank n holds the same node sequences on both sides (equal scores can come in any order;
    compared as multisets, since two choice sets can give the same tree);
  * in the run cut by rank n (it may continue past n), every derivation is a real derivation of the forest with its
    stated score, the score recomputed from the rule weights by walking the forest.
"""
import heapq
import math
import re
import sys

import numpy as np

TOKEN = re.compile(r"#\d+\(|#\d+|\(|\)|OR|\d+")


def forests_to_arrays(texts):
    """forest-em text forests -> (node_off, next, label, backref) as cml_forest_batch holds them (ForestSet::read)"""
    node_off, nxt, label, backref = [0], [], [], []
    for text in texts:
        nx, lb, br, stack, defs, pending = [], [], [], [], {}, None
        toks = TOKEN.findall(text)
        i = 0
        while i < len(toks):
            t = toks[i]
            if t.endswith("(") and t.startswith("#"):
                pending = int(t[1:-1])
                t = "("
            if t == "(":
                j = len(nx)
                if pending is not None:
                    defs[pending], pending = j, None
                head = toks[i + 1]
                nx.append(0)
                lb.append(0 if head == "OR" else int(head))
                br.append(0)
                stack.append(j)
                i += 2
                continue
            if t == ")":
                nx[stack.pop()] = len(nx)
            elif t.startswith("#"):
                nx.append(len(nx) + 1)
                lb.append(defs[int(t[1:])])
                br.append(1)
            else:
                nx.append(len(nx) + 1)
                lb.append(int(t))
                br.append(0)
            i += 1
        assert not stack, text
        nxt += nx
        label += lb
        backref += br
        node_off.append(node_off[-1] + len(nx))
    return (np.array(node_off, np.uint64), np.array(nxt, np.uint32), np.array(label, np.uint32),
            np.array(backref, np.uint8))


class ForestRef:
    """one forest's pre-order arrays and the rule weights (ln): its k best derivations, and the score of a node sequence"""

    def __init__(self, nxt, label, backref, ln_w):
        self.nx, self.lb, self.br = [int(x) for x in nxt], [int(x) for x in label], [int(x) for x in backref]
        self.ln_w = np.asarray(ln_w, np.float64)
        n = len(self.nx)
        self.slots = [[] for _ in range(n)]  # real node -> its child slots, resolved to real nodes
        for p in range(n):
            if not self.br[p]:
                q = p + 1
                while q < self.nx[p]:
                    self.slots[p].append(self.lb[q] if self.br[q] else q)
                    q = self.nx[q]
        self.D = [None] * n      # derivations found so far: (score, back pointer)
        self.heap = [None] * n
        self.seen = [None] * n
        sys.setrecursionlimit(max(sys.getrecursionlimit(), 20 * n + 1000))

    def _and_score(self, v, ranks):
        s = float(self.ln_w[self.lb[v]])
        for c, j in zip(self.slots[v], ranks):
            s = s + self.D[c][j][0]
        return s

    def _push(self, v, cand):
        if self.lb[v]:
            sc = self._and_score(v, cand)
        else:
            q, j = cand
            sc = self.D[self.slots[v][q]][j][0]
        if sc > -math.inf:
            heapq.heappush(self.heap[v], (-sc, cand))

    def get(self, v, r):
        """does real node v have an r-th derivation?"""
        if self.D[v] is None:
            self.D[v], self.heap[v], self.seen[v] = [], [], set()
            if self.lb[v]:
                z = tuple(0 for _ in self.slots[v])
                if all(self.get(c, 0) for c in self.slots[v]):
                    self.seen[v].add(z)
                    self._push(v, z)
            else:
                for q, c in enumerate(self.slots[v]):
                    if self.get(c, 0):
                        self._push(v, (q, 0))
        while len(self.D[v]) <= r and self.heap[v]:
            nsc, cand = heapq.heappop(self.heap[v])
            self.D[v].append((-nsc, cand))
            if self.lb[v]:
                for i, c in enumerate(self.slots[v]):
                    nb = cand[:i] + (cand[i] + 1,) + cand[i + 1:]
                    if nb not in self.seen[v] and self.get(c, cand[i] + 1):
                        self.seen[v].add(nb)
                        self._push(v, nb)
            else:
                q, j = cand
                if self.get(self.slots[v][q], j + 1):
                    self._push(v, (q, j + 1))
        return r < len(self.D[v])

    def nodes(self, v, r):
        out = []
        while not self.lb[v]:
            q, j = self.D[v][r][1]
            v, r = self.slots[v][q], j
        out.append(v)
        for c, j in zip(self.slots[v], self.D[v][r][1]):
            out.extend(self.nodes(c, j))
        return out

    def kbest(self, k):
        """[(score, node tuple)] * k, best first; (-inf, ()) past the last derivation"""
        return [(self.D[0][r][0], tuple(self.nodes(0, r))) if self.get(0, r) else (-math.inf, ()) for r in range(k)]

    def score_of(self, seq):
        """ln score of a node sequence, or None if it is not a derivation of the forest"""
        pos = [0]

        def reach(c, x):  # can slot node c (real) stand for AND node x?
            if self.lb[c]:
                return c == x
            return any(reach(d, x) for d in self.slots[c])

        def derive(c):
            if pos[0] >= len(seq):
                return None
            x = seq[pos[0]]
            if not (0 <= x < len(self.nx)) or self.br[x] or not self.lb[x] or not reach(c, x):
                return None
            pos[0] += 1
            s = float(self.ln_w[self.lb[x]])
            for d in self.slots[x]:
                t = derive(d)
                if t is None:
                    return None
                s = s + t
            return s

        s = derive(0)
        return s if s is not None and pos[0] == len(seq) else None

    def tree(self, seq):
        """the -v tree text of a node sequence: '(rule child ...)', a leaf rule bare"""
        it = iter(seq)

        def rec():
            x = next(it)
            if not self.slots[x]:
                return str(self.lb[x])
            return "(" + str(self.lb[x]) + "".join(" " + rec() for _ in self.slots[x]) + ")"
        return rec()


def forest_refs(node_off, nxt, label, backref, ln_w):
    return [ForestRef(nxt[int(node_off[i]):int(node_off[i + 1])], label[int(node_off[i]):int(node_off[i + 1])],
                      backref[int(node_off[i]):int(node_off[i + 1])], ln_w) for i in range(len(node_off) - 1)]


def read_kbest_forests(path, k):
    """-v --kbest=k file -> [[(ln score, ln sum, tree text) * k] per forest]"""
    from forest_helpers import parse_ln
    rows = []
    for ln in open(path).read().split("\n")[:-1]:
        head, tree = ln.split("% ", 1)
        best, total = (parse_ln(t) for t in head.split("=")[0].split("/"))
        rows.append((best, total, tree))
    assert len(rows) % k == 0, (len(rows), k)
    return [rows[i:i + k] for i in range(0, len(rows), k)]


def _close(a, b, rel):
    return a == b or abs(a - b) <= rel * max(1.0, abs(a), abs(b))


def compare_kbest(want, got, score_of=None, run_of=None, tol=1e-9):
    """apply the comparison rule to one forest's lists (want = reference, got = checked side, same length n) of
    (score, derivation) pairs.  The run cut by rank n is checked by score_of(derivation) -> ln score or None, or by
    run_of(r) -> every derivation of the reference's run starting at rank r (when derivations are tree texts)."""
    k = len(want)
    assert len(got) == k
    for r, ((ww, _), (gw, gp)) in enumerate(zip(want, got)):
        if ww == -math.inf or gw == -math.inf:
            assert ww == gw == -math.inf, (r, ww, gw)
            assert not gp, (r, gp)
        else:
            assert _close(ww, gw, tol), (r, ww, gw)
    r = 0
    while r < k and want[r][0] > -math.inf:
        end = r + 1
        while end < k and want[end][0] > -math.inf and _close(want[end][0], want[r][0], 1e-12):
            end += 1
        if end < k:
            assert sorted(p for _, p in want[r:end]) == sorted(p for _, p in got[r:end]), (r, end, want[r:end], got[r:end])
        else:
            if score_of is not None:
                for w, p in got[r:end]:
                    pw = score_of(p)
                    assert pw is not None and _close(pw, w, tol), (r, p, pw, w)
            if run_of is not None:
                pool = list(run_of(r))
                for _, p in got[r:end]:
                    assert p in pool, (r, p)
                    pool.remove(p)
        r = end
