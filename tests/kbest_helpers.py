"""k-best derivation lists (carmel-b200 --viterbi=FILE -k n): reading the files, the CPU reference the parity tests and
bench_kbest.py hold the GPU to, and the comparison rule they apply.

The reference (Lattices.kbest) works on the lattices the CPU oracle builds (carmel_oracle --dump-trellis: the
reference's state ids and stored arc lists) with the oracle's arc weights (--dump-estimate), and uses a different
algorithm from the GPU: a lazy enumeration with a candidate heap per state (Huang & Chiang 2005, "Better k-best
parsing", algorithm 3) instead of an eager k-way merge in layered order.

Comparison rule, rank by rank over the n lines of an example:
  * weights agree within 1e-9 * max(1, |w|); padding (-inf) on both sides;
  * ranks are grouped into runs of equal weight (within 1e-12 relative);
  * every run that ends before rank n holds the same SET of arc-id sequences on both sides (equal weights can come in
    any order);
  * in the run cut by rank n (it may continue past n), every path is a real derivation of that weight.
"""
import heapq
import math
import sys

import numpy as np


def read_kbest(path, k):
    """[[(ln_w, [arc ids]) * k] per example] from a file with k lines per example"""
    rows = []
    for ln in open(path):
        head = ln.split("|")[0].split()
        rows.append((float(head[0]), tuple(int(x) for x in head[2:2 + int(head[1])])))
    assert len(rows) % k == 0, (len(rows), k)
    return [rows[i:i + k] for i in range(0, len(rows), k)]


class Lattices:
    """the lattices of a --dump-trellis file and the arc-table ln weights of a --dump-estimate file: is an arc-id
    sequence a start -> goal path of example e, and what is its weight"""

    def __init__(self, trellis, ln_w):
        self.t, self.ln_w = trellis, np.asarray(ln_w, np.float64)
        self.rows, row, arc = [], 0, 0
        for e in range(trellis["n_ex"]):
            n = int(trellis["ex_states"][e])
            off = trellis["arc_off"][row:row + n + 1].astype(np.int64) + arc
            self.rows.append(off)
            row += n + 1
            arc = int(off[-1])

    def weight(self, e, ids):
        """ln weight of the path, or None if ids is not a start -> goal path of example e"""
        off, dst, aid = self.rows[e], self.t["arc_dst"], self.t["arc_id"]
        s, w = 0, 0.0
        for a in ids:
            nxt = [k for k in range(off[s], off[s + 1]) if aid[k] == a]
            if not nxt:
                return None
            s = int(dst[nxt[0]])
            w += self.ln_w[a]
        return w if s == int(self.t["ex_fin"][e]) else None

    def paths(self, e, limit=200000):
        """every start -> goal path of example e as (ln weight, arc ids)"""
        off, dst, aid, fin = self.rows[e], self.t["arc_dst"], self.t["arc_id"], int(self.t["ex_fin"][e])
        out, stack, n = [], [(0, 0.0, ())], 0
        while stack:
            s, w, ids = stack.pop()
            if s == fin:
                out.append((w, ids))
            for k in range(off[s], off[s + 1]):
                n += 1
                assert n < limit, "lattice too large for enumeration"
                stack.append((int(dst[k]), w + self.ln_w[aid[k]], ids + (int(aid[k]),)))
        return out

    def kbest(self, e, k):
        """the k best derivations of example e, best first, as (ln weight, arc ids); (-inf, ()) past the last one.
        A state's r-th derivation is computed only when asked for: each state keeps a heap of candidates (in-arc,
        rank of the source's derivation); taking candidate (a, j) pushes (a, j + 1), which asks the source for its
        (j + 1)-th derivation in turn.  Derivations of weight zero are never listed."""
        off, dst, aid, fin = self.rows[e], self.t["arc_dst"], self.t["arc_id"], int(self.t["ex_fin"][e])
        n = len(off) - 1
        inl = [[] for _ in range(n)]  # in-arcs (source, arc id, ln weight), sources in id order, stored arc order
        for s in range(n):
            for q in range(off[s], off[s + 1]):
                inl[int(dst[q])].append((s, int(aid[q]), float(self.ln_w[aid[q]])))
        sys.setrecursionlimit(max(sys.getrecursionlimit(), 4 * n + 1000))  # get() recurses along a path
        D = [[] for _ in range(n)]  # derivations found so far: (ln weight, in-arc, source rank)
        D[0].append((0.0, -1, -1))
        heap, started = [[] for _ in range(n)], [False] * n

        def push(v, a, j):
            sc = D[inl[v][a][0]][j][0] + inl[v][a][2]
            if sc > -math.inf:
                heapq.heappush(heap[v], (-sc, a, j))

        def get(v, r):  # does state v have an r-th derivation?
            if r < len(D[v]):
                return True
            if v == 0:
                return False
            if not started[v]:
                started[v] = True
                for a in range(len(inl[v])):
                    if get(inl[v][a][0], 0):
                        push(v, a, 0)
            while len(D[v]) <= r and heap[v]:
                nsc, a, j = heapq.heappop(heap[v])
                D[v].append((-nsc, a, j))
                if get(inl[v][a][0], j + 1):
                    push(v, a, j + 1)
            return r < len(D[v])

        out = []
        for r in range(k):
            if not get(fin, r):
                out.append((-math.inf, ()))
                continue
            ids, v, j = [], fin, r
            while v != 0:
                _, a, jj = D[v][j]
                ids.append(inl[v][a][1])
                v, j = inl[v][a][0], jj
            out.append((D[fin][r][0], tuple(reversed(ids))))
        return out


def _close(a, b, rel):
    return a == b or abs(a - b) <= rel * max(1.0, abs(a), abs(b))


def compare_kbest(want, got, weight_of=None):
    """apply the comparison rule to one example's lists (want = reference, got = checked side, same length k).
    weight_of(ids) -> ln weight of a real derivation or None; needed to check the run cut by rank k."""
    k = len(want)
    assert len(got) == k
    for r, ((ww, _), (gw, gp)) in enumerate(zip(want, got)):
        if ww == -math.inf or gw == -math.inf:
            assert ww == gw == -math.inf, (r, ww, gw)
            assert not gp, (r, gp)
        else:
            assert _close(ww, gw, 1e-9), (r, ww, gw)
    r = 0
    while r < k and want[r][0] > -math.inf:
        end = r + 1
        while end < k and want[end][0] > -math.inf and _close(want[end][0], want[r][0], 1e-12):
            end += 1
        if end < k:
            assert {p for _, p in want[r:end]} == {p for _, p in got[r:end]}, (r, end, want[r:end], got[r:end])
        else:
            assert len({p for _, p in got[r:end]}) == end - r, ("repeated path", got[r:end])
            if weight_of is not None:
                for w, p in got[r:end]:
                    pw = weight_of(p)
                    assert pw is not None and _close(pw, w, 1e-9), (r, p, pw, w)
        r = end
