"""Decoding new strings with the other tape free (carmel-b200 --decode=FILE --given=input|output, cml_build_free_trellises):
the CPU reference the parity tests and bench_decode.py hold the GPU to.

The reference builds the lattice of include/carmel_b200.h ("lattices of one given string, the other tape free") with a
different algorithm from k_build_free: a memoised recursion over (machine state, position) for co-reachability, a
depth-first walk from (start, 0) for reachability, then a sort of the kept pairs into the (position, eps-level, state)
numbering.  Its result has the dict shape kbest_helpers.Lattices takes, so Lattices.kbest and compare_kbest (the
comparison rule of the --viterbi -k tests) apply unchanged.

Machines are dicts of arc-table arrays: n_states, final_state, state_arc_off, arc_in, arc_out, arc_dest (start = state
0, symbol 0 = *e*), plus `names` (symbol id -> spelling) when they come from carmel text.
"""
import math
import re
import subprocess
import sys

import numpy as np

from kbest_helpers import Lattices

_TOK = re.compile(r'"(?:[^"\\]|\\.)*"|\(|\)|[^\s()]+')


class GivenEpsCycle(ValueError):
    """the arcs with *e* on the given tape form a cycle"""


def _is_label(tok):
    return tok.startswith('"') or tok == "*e*"


def parse_wfst(text, alphabet=None):
    """carmel text -> arc-table arrays.  States are numbered by first appearance as a source in file order (the source
    of the first arc is the start, state 0), then the states that only appear as destinations or as the final state.
    Arc ids follow the file order state by state, which is the arc-table order of a machine written by --write-composed.
    alphabet: a shared {spelling: id} dict (*e* = 0), extended as needed."""
    alphabet = {"*e*": 0} if alphabet is None else alphabet
    toks = _TOK.findall(re.sub(r"(?m)^\s*%.*$", "", text))
    final, i, arcs = toks[0], 1, []
    while i < len(toks):
        assert toks[i] == "(", toks[i:i + 6]
        src = toks[i + 1]
        j = i + 2
        while toks[j] == "(":  # one or more (dst labels [weight]) groups
            dst, k, labels = toks[j + 1], j + 2, []
            while toks[k] != ")":
                if _is_label(toks[k]):
                    labels.append(toks[k])
                k += 1
            assert 1 <= len(labels) <= 2, toks[j:k + 1]
            lin, lout = labels[0], labels[-1]
            arcs.append((src, dst, lin, lout))
            j = k + 1
        assert toks[j] == ")", toks[i:j + 1]
        i = j + 1
    idx = {}
    for s, _, _, _ in arcs:
        idx.setdefault(s, len(idx))
    for _, d, _, _ in arcs:
        idx.setdefault(d, len(idx))
    idx.setdefault(final, len(idx))
    sym = lambda t: alphabet.setdefault(t, len(alphabet))
    by_src = [[] for _ in idx]
    for a in arcs:
        by_src[idx[a[0]]].append(a)
    arcs = [a for lst in by_src for a in lst]  # (a state's arcs may be spread over the file)
    off = np.zeros(len(idx) + 1, np.uint32)
    off[1:] = np.cumsum([len(lst) for lst in by_src])
    m = dict(n_states=len(idx), final_state=idx[final], state_arc_off=off,
             arc_in=np.array([sym(a[2]) for a in arcs], np.uint32), arc_out=np.array([sym(a[3]) for a in arcs], np.uint32),
             arc_dest=np.array([idx[a[1]] for a in arcs], np.uint32), alphabet=alphabet)
    m["names"] = {v: k for k, v in alphabet.items()}
    return m


def symbols(line, alphabet):
    """a strings-file line -> symbol ids (unknown spellings get new ids, which no arc carries)"""
    return [alphabet.setdefault(t, len(alphabet)) for t in _TOK.findall(line)]


def eps_levels(m, given):
    """longest-path depth of every state in the subgraph of the arcs with *e* on the given tape"""
    glab = m["arc_in"] if given == 0 else m["arc_out"]
    off, dst, Q = m["state_arc_off"], m["arc_dest"], m["n_states"]
    succ = [[int(dst[a]) for a in range(off[q], off[q + 1]) if glab[a] == 0] for q in range(Q)]
    pred = [[] for _ in range(Q)]
    for q in range(Q):
        for d in succ[q]:
            pred[d].append(q)
    level, state = [0] * Q, [0] * Q  # 0 new, 1 on the path, 2 done

    def depth(q):
        if state[q] == 1:
            raise GivenEpsCycle(f"state {q}")
        if state[q] == 0:
            state[q] = 1
            level[q] = max([depth(p) + 1 for p in pred[q]], default=0)
            state[q] = 2
        return level[q]

    sys.setrecursionlimit(max(sys.getrecursionlimit(), 4 * Q + 1000))
    for q in range(Q):
        depth(q)
    return level


def free_lattices(m, strings, given):
    """the lattices of `strings` (lists of symbol ids on tape `given`) with the other tape free: a dict in the shape of
    a --dump-trellis batch (n_ex, ex_states, ex_fin, ex_weight, arc_off, arc_dst, arc_id) plus kept / dropped string
    indices.  Raises GivenEpsCycle."""
    level = eps_levels(m, given)
    glab = m["arc_in"] if given == 0 else m["arc_out"]
    off, dst, fin = m["state_arc_off"], m["arc_dest"], int(m["final_state"])
    by_sym = []  # per state: given symbol -> [(arc, destination)] in arc-table order
    for q in range(m["n_states"]):
        by_sym.append({})
        for a in range(off[q], off[q + 1]):
            by_sym[q].setdefault(int(glab[a]), []).append((a, int(dst[a])))
    out = dict(ex_states=[], ex_fin=[], arc_off=[], arc_dst=[], arc_id=[], kept=[], dropped=[])
    for e, s in enumerate(strings):
        n = len(s)
        memo = {}

        def step(q, t):  # (arc, next cell) of every arc leaving (q, t), in arc-table order
            r = [(a, (d, t)) for a, d in by_sym[q].get(0, ())]
            if t < n and s[t] != 0:
                r += [(a, (d, t + 1)) for a, d in by_sym[q].get(s[t], ())]
            return sorted(r)

        def coreach(q, t):
            if (q, t) not in memo:
                memo[(q, t)] = (q == fin and t == n) or any([coreach(*c) for _, c in step(q, t)])
            return memo[(q, t)]

        sys.setrecursionlimit(max(sys.getrecursionlimit(), 4 * (n + 1) * len(by_sym) + 1000))
        if not coreach(0, 0):
            out["dropped"].append(e)
            continue
        kept, stack = {(0, 0)}, [(0, 0)]
        while stack:
            c = stack.pop()
            for _, d in step(*c):
                if d not in kept and coreach(*d):
                    kept.add(d)
                    stack.append(d)
        cells = sorted(kept, key=lambda c: (c[1], level[c[0]], c[0]))
        num = {c: i for i, c in enumerate(cells)}
        row, base = [0], len(out["arc_dst"])
        for c in cells:
            for a, d in step(*c):
                if d in num:
                    out["arc_dst"].append(num[d])
                    out["arc_id"].append(a)
            row.append(len(out["arc_dst"]) - base)
        out["arc_off"].append(np.asarray(row, np.uint32))
        out["ex_states"].append(len(cells))
        out["ex_fin"].append(num[(fin, n)])
        out["kept"].append(e)
    u32 = lambda x: np.asarray(x, np.uint32)
    return dict(n_ex=len(out["kept"]), ex_states=u32(out["ex_states"]), ex_fin=u32(out["ex_fin"]),
                ex_weight=np.ones(len(out["kept"])), arc_off=np.concatenate(out["arc_off"]).astype(np.uint32)
                if out["arc_off"] else u32([]), arc_dst=u32(out["arc_dst"]), arc_id=u32(out["arc_id"]),
                kept=u32(out["kept"]), dropped=u32(out["dropped"]))


def longest_path(lat, e):
    """arcs on the longest start -> goal path of lattice e of a free_lattices batch (its states are in topological
    order)"""
    L = Lattices(lat, np.zeros(1))
    offs, d = L.rows[e], lat["arc_dst"]
    best = [-1] * (len(offs) - 1)
    best[0] = 0
    for s in range(len(offs) - 1):
        if best[s] >= 0:
            for k in range(offs[s], offs[s + 1]):
                best[int(d[k])] = max(best[int(d[k])], best[s] + 1)
    return best[int(lat["ex_fin"][e])]


def decoded_string(m, ids, given):
    """the free-tape labels of a path's arcs, *e* dropped, spelled as the model spells them"""
    free = m["arc_out"] if given == 0 else m["arc_in"]
    return " ".join(m["names"][int(free[a])] for a in ids if free[a] != 0)


def read_decode(path, k):
    """[[(ln_w, arc ids, decoded string)] * k per string] of a --decode file"""
    rows = []
    for ln in open(path):
        head, _, tail = ln.rstrip("\n").partition(" ||")
        f = head.split("|")[0].split()
        rows.append((float(f[0]), tuple(int(x) for x in f[2:2 + int(f[1])]), tail.strip()))
    assert len(rows) % k == 0, (len(rows), k)
    return [rows[i:i + k] for i in range(0, len(rows), k)]


def reference_model(oracle_bin, tmp, args):
    """the composed machine of a carmel-b200 command line (`args`: flags and transducer files, no corpus) as the CPU
    oracle composes it, with its arc-table ln weights after the initial normalisation (--dump-estimate)"""
    from helpers import read_estimate_dump
    flags = [a for a in args if a.startswith("-")]
    files = [a for a in args if not a.startswith("-")]
    open(f"{tmp}/empty.data", "w").close()
    p = subprocess.run([oracle_bin, *(flags or ["-t"]), f"--write-composed={tmp}/ref.fst", f"--dump-estimate={tmp}/ref.e",
                        f"{tmp}/empty.data", *files], capture_output=True, text=True)
    assert p.returncode == 0, p.stderr
    m = parse_wfst(open(f"{tmp}/ref.fst").read())
    m["ln_w"] = read_estimate_dump(f"{tmp}/ref.e")["ln_w"]
    assert m["ln_w"].size == m["arc_in"].size, (m["ln_w"].size, m["arc_in"].size)
    return m


def random_machine(rng, n_states=4, n_in=3, n_out=3, density=0.5, eps_rate=0.25, in_prefix="i", out_prefix="o"):
    """(arc-table arrays, carmel text): state 0 is the start, the last state final; every arc with *e* on either tape
    goes to a later state, so the machine has no given-*e* cycle whichever tape is given.  Input symbols are
    <in_prefix>0.. and output symbols <out_prefix>0.. (ids 1..n_in and n_in+1.. in the arrays)"""
    arcs = [(k, k + 1, 1 + k % n_in, 1 + n_in + k % n_out) for k in range(n_states - 1)]
    for s in range(n_states):
        for d in range(n_states):
            if rng.random() > density:
                continue
            for _ in range(1 + int(rng.integers(0, 3))):
                i = 0 if rng.random() < eps_rate else 1 + int(rng.integers(0, n_in))
                o = 0 if rng.random() < eps_rate else 1 + n_in + int(rng.integers(0, n_out))
                if (i == 0 or o == 0) and d <= s:
                    continue
                arcs.append((s, d, i, o))
    arcs.sort(key=lambda a: a[0])  # (stable: arcs of a state keep their order)
    w = rng.uniform(0.05, 1.0, len(arcs))
    names = ["*e*"] + [f'"{in_prefix}{k}"' for k in range(n_in)] + [f'"{out_prefix}{k}"' for k in range(n_out)]
    off = np.zeros(n_states + 1, np.uint32)
    for a in arcs:
        off[a[0] + 1] += 1
    m = dict(n_states=n_states, final_state=n_states - 1, state_arc_off=np.cumsum(off).astype(np.uint32),
             arc_in=np.array([a[2] for a in arcs], np.uint32), arc_out=np.array([a[3] for a in arcs], np.uint32),
             arc_dest=np.array([a[1] for a in arcs], np.uint32), names=dict(enumerate(names)),
             alphabet={n: i for i, n in enumerate(names)})
    lines = [f"q{n_states - 1}"] + [f"(q{s} (q{d} {names[i]} {names[o]} {x:.6g}))" for (s, d, i, o), x in zip(arcs, w)]
    return m, "\n".join(lines) + "\n"


def reference_kbest(m, strings, given, k, lat=None):
    """[k * (ln_w, arc ids, decoded string)] per string: the reference lattice's k best derivations at m["ln_w"];
    (-inf, (), "") past the last one and for strings without a derivation.  `lat`: free_lattices(m, strings, given)
    when the caller has built it already.  Returns (lists, lattices, Lattices)."""
    lat = free_lattices(m, strings, given) if lat is None else lat
    L = Lattices(lat, m["ln_w"])
    lists = [[(-math.inf, (), "")] * k for _ in strings]
    for i, e in enumerate(lat["kept"]):
        lists[int(e)] = [(w, p, decoded_string(m, p, given)) for w, p in L.kbest(i, k)]
    return lists, lat, L
