"""ctypes binding of the forest-em part of include/carmel_b200.h (cml_forests_*, cml_forest_job_*).

Plumbing for tests and bench.py; the product is the CUDA library.  No CPU fallback."""
from __future__ import annotations

import ctypes as C

import numpy as np

from .api import ALLREDUCE_FN, CarmelB200Error, load_library

ZERO, SKIP, UNIFORM = 0, 1, 2
_vp = C.c_void_p
_u64p = C.POINTER(C.c_uint64)
_u32p = C.POINTER(C.c_uint32)
_u8p = C.POINTER(C.c_uint8)
_f64p = C.POINTER(C.c_double)


class CmlForestBatch(C.Structure):
    _fields_ = [("n_forests", C.c_uint64), ("node_off", _u64p), ("next", _u32p), ("label", _u32p), ("backref", _u8p)]


class CmlForestEstimateResult(C.Structure):
    _fields_ = [("sum_ln_p", C.c_double), ("n_zero", C.c_uint64), ("n_forests", C.c_uint64)]


class CmlForestNormOpts(C.Structure):
    _fields_ = [("prior_total", C.c_double), ("add_k", C.c_double), ("zero_mode", C.c_int)]


class CmlForestJobInfo(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("forests", "nodes", "hyperedges", "links", "rulespace", "iterations")] + [
        ("best_avg_logprob", C.c_double)]


_bound = False


def _lib():
    global _bound
    lib = load_library()
    if not _bound:
        lib.cml_forests_create.argtypes = [C.POINTER(_vp), C.c_int, C.c_int]
        lib.cml_forests_destroy.argtypes = [_vp]
        lib.cml_forests_destroy.restype = None
        lib.cml_forests_last_error.argtypes = [_vp]
        lib.cml_forests_last_error.restype = C.c_char_p
        lib.cml_forests_set_stream.argtypes = [_vp, _vp]
        lib.cml_forests_set_layout.argtypes = [_vp, C.c_int]
        lib.cml_forests_layout_stats.argtypes = [_vp] + [_u64p] * 5
        lib.cml_forests_level_stats.argtypes = [_vp] + [_u64p] * 6
        lib.cml_forests_launch_count.argtypes = [_vp]
        lib.cml_forests_launch_count.restype = C.c_uint64
        lib.cml_forests_set_rules.argtypes = [_vp, C.c_uint64, C.c_uint64, _u64p, _u64p]
        lib.cml_forests_set_params.argtypes = [_vp, _f64p]
        lib.cml_forests_get_params.argtypes = [_vp, _f64p]
        lib.cml_forests_add.argtypes = [_vp, C.POINTER(CmlForestBatch)]
        lib.cml_forests_totals.argtypes = [_vp] + [_u64p] * 4
        lib.cml_forests_estimate.argtypes = [_vp, C.POINTER(CmlForestEstimateResult)]
        lib.cml_forests_estimate_launch.argtypes = [_vp]
        lib.cml_forests_estimate_finish.argtypes = [_vp, C.POINTER(CmlForestEstimateResult)]
        lib.cml_forests_last_time_ms.argtypes = [_vp, C.POINTER(C.c_float), _u32p]
        lib.cml_forests_get_inside.argtypes = [_vp, _f64p, C.c_uint64]
        lib.cml_forests_get_counts.argtypes = [_vp, _f64p, C.c_uint64]
        lib.cml_forests_reduce_buffer.argtypes = [_vp, C.POINTER(_vp), _u64p]
        lib.cml_forests_comm_init_rank.argtypes = [_vp, C.c_int, C.c_int, C.c_char_p]
        lib.cml_forests_allreduce_counts.argtypes = [_vp]
        lib.cml_forests_maximize.argtypes = [_vp, C.POINTER(CmlForestNormOpts), _f64p, _u64p]
        lib.cml_forests_normalize_params.argtypes = [_vp]
        lib.cml_forests_viterbi.argtypes = [_vp, C.POINTER(CmlForestBatch), _f64p, _u32p]
        lib.cml_forests_kbest.argtypes = [_vp, C.POINTER(CmlForestBatch), C.c_uint32, _f64p, _u32p, _u64p, _u32p, C.c_uint64]
        lib.cml_forests_set_kbest_scratch_mb.argtypes = [_vp, C.c_uint64]
        lib.cml_forests_kbest_stats.argtypes = [_vp, _u64p, _u64p, C.POINTER(C.c_float)]
        lib.cml_forests_sample.argtypes = [_vp, C.POINTER(CmlForestBatch), C.c_uint32, C.c_uint64, _u64p, _f64p, _u32p,
                                           _u64p, _u32p, C.c_uint64, _f64p]
        lib.cml_forests_sample_stats.argtypes = [_vp, _u64p, _u64p, C.POINTER(C.c_float)]
        lib.cml_forest_job_open.argtypes = [C.POINTER(_vp), C.c_int, C.POINTER(C.c_char_p)]
        lib.cml_forest_job_close.argtypes = [_vp]
        lib.cml_forest_job_close.restype = None
        lib.cml_forest_job_error.argtypes = [_vp]
        lib.cml_forest_job_error.restype = C.c_char_p
        lib.cml_forest_job_set_allreduce.argtypes = [_vp, ALLREDUCE_FN, _vp]
        lib.cml_forest_job_prepare.argtypes = [_vp]
        lib.cml_forest_job_context.argtypes = [_vp]
        lib.cml_forest_job_context.restype = _vp
        lib.cml_forest_job_train.argtypes = [_vp]
        lib.cml_forest_job_write.argtypes = [_vp]
        lib.cml_forest_job_stats.argtypes = [_vp, C.POINTER(CmlForestJobInfo)]
        _bound = True
    return lib


def _arr(a, dtype):
    return np.ascontiguousarray(a, dtype=dtype)


class Forests:
    """One cml_forests handle: rules + parameters + resident forests of one GPU."""

    def __init__(self, device: int = 0, precision: int = 32, handle=None):
        self.lib = _lib()
        self._own = handle is None
        if handle is None:
            h = _vp()
            rc = self.lib.cml_forests_create(C.byref(h), device, precision)
            if rc != 0:
                raise CarmelB200Error(rc, self.lib.cml_forests_last_error(None).decode())
            handle = h
        self.h = handle
        self.rulespace = 0

    def close(self):
        if self._own and self.h:
            self.lib.cml_forests_destroy(self.h)
        self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ok(self, rc):
        if rc != 0:
            raise CarmelB200Error(rc, self.lib.cml_forests_last_error(self.h).decode())

    def set_stream(self, cuda_stream: int):
        self._ok(self.lib.cml_forests_set_stream(self.h, _vp(cuda_stream)))

    def set_layout(self, layout: int):
        """0 auto, 1 warp/CTA per forest, 2 thread per forest, 3 level-synchronous tiles (CTA per run of forests)"""
        self._ok(self.lib.cml_forests_set_layout(self.h, layout))

    def layout_stats(self) -> dict:
        v = [C.c_uint64() for _ in range(5)]
        self._ok(self.lib.cml_forests_layout_stats(self.h, *[C.byref(x) for x in v]))
        return dict(zip(("tile_forests", "tiles", "steps", "padded_steps", "padded_rows"), (x.value for x in v)))

    def level_stats(self) -> dict:
        v = [C.c_uint64() for _ in range(6)]
        self._ok(self.lib.cml_forests_level_stats(self.h, *[C.byref(x) for x in v]))
        return dict(zip(("level_forests", "level_tiles", "level_nodes", "level_links", "max_tile_nodes", "small_tiles"),
                        (x.value for x in v)))

    def set_rules(self, rulespace: int, group_off, group_members):
        go, gm = _arr(group_off, np.uint64), _arr(group_members, np.uint64)
        self._ok(self.lib.cml_forests_set_rules(self.h, rulespace, len(go) - 1, go.ctypes.data_as(_u64p), gm.ctypes.data_as(_u64p)))
        self.rulespace = rulespace

    def set_params(self, ln_w):
        w = _arr(ln_w, np.float64)
        assert len(w) == self.rulespace
        self._ok(self.lib.cml_forests_set_params(self.h, w.ctypes.data_as(_f64p)))

    def get_params(self) -> np.ndarray:
        w = np.empty(self.rulespace, np.float64)
        self._ok(self.lib.cml_forests_get_params(self.h, w.ctypes.data_as(_f64p)))
        return w

    @staticmethod
    def _batch(node_off, nxt, label, backref):
        """(cml_forest_batch, the contiguous arrays it points into: keep them alive while the batch is used)"""
        no, nx, lb, br = _arr(node_off, np.uint64), _arr(nxt, np.uint32), _arr(label, np.uint32), _arr(backref, np.uint8)
        b = CmlForestBatch(len(no) - 1, no.ctypes.data_as(_u64p), nx.ctypes.data_as(_u32p), lb.ctypes.data_as(_u32p),
                           br.ctypes.data_as(_u8p))
        return b, (no, nx, lb, br)

    def add(self, node_off, nxt, label, backref):
        b, keep = self._batch(node_off, nxt, label, backref)
        self._ok(self.lib.cml_forests_add(self.h, C.byref(b)))

    def viterbi(self, node_off, nxt, label, backref):
        """best derivation of every forest of the batch (cml_forests_viterbi): (ln score [n_forests], chosen child of
        every OR node [n_nodes]: in-forest pre-order index, 0xFFFFFFFF elsewhere)"""
        b, keep = self._batch(node_off, nxt, label, backref)
        n = int(keep[0][-1])
        root, best = np.empty(max(b.n_forests, 1)), np.empty(max(n, 1), np.uint32)
        self._ok(self.lib.cml_forests_viterbi(self.h, C.byref(b), root.ctypes.data_as(_f64p), best.ctypes.data_as(_u32p)))
        return root[:b.n_forests], best[:n]

    def kbest(self, k: int, node_off, nxt, label, backref, nodes: bool = True, cap: int | None = None):
        """the k best derivations of every forest of the batch (cml_forests_kbest): (ln_score [n_forests, k],
        n_and [n_forests, k], base [n_forests * k + 1], nodes); derivation (i, r) is nodes[base[i*k+r]:][:n_and[i, r]],
        in-forest pre-order indices of its AND nodes.  nodes=False asks for scores and sizes only (nodes is None).
        cap: size of the node buffer handed to the library (default: k * n_nodes, grown once if that is too small)."""
        b, keep = self._batch(node_off, nxt, label, backref)
        nf, n = b.n_forests, int(keep[0][-1])
        score, lens = np.empty(max(nf * k, 1)), np.empty(max(nf * k, 1), np.uint32)
        base = np.zeros(nf * k + 1, np.uint64)

        def call(buf, c):
            return self.lib.cml_forests_kbest(self.h, C.byref(b), k, score.ctypes.data_as(_f64p), lens.ctypes.data_as(_u32p),
                                              base.ctypes.data_as(_u64p), buf.ctypes.data_as(_u32p) if buf is not None else None, c)
        out = None
        if nodes:
            c = k * n if cap is None else cap
            out = np.empty(max(c, 1), np.uint32)
            rc = call(out, c)
            if rc == -1 and cap is None and int(base[-1]) > c:
                c = int(base[-1])
                out = np.empty(max(c, 1), np.uint32)
                rc = call(out, c)
            self._ok(rc)
            out = out[:int(base[-1])]
        else:
            self._ok(call(None, 0))
        return score[:nf * k].reshape(nf, k), lens[:nf * k].reshape(nf, k), base, out

    def set_kbest_scratch_mb(self, mb: int):
        self._ok(self.lib.cml_forests_set_kbest_scratch_mb(self.h, mb))

    def _decode_stats(self, fn) -> dict:
        b, c, ms = C.c_uint64(), C.c_uint64(), C.c_float()
        self._ok(fn(self.h, C.byref(b), C.byref(c), C.byref(ms)))
        return {"scratch_bytes": b.value, "chunks": c.value, "kernel_ms": ms.value}

    def kbest_stats(self) -> dict:
        """the last kbest() call: scratch bytes of its largest chunk, chunks, kernel time (CUDA events, ms)"""
        return self._decode_stats(self.lib.cml_forests_kbest_stats)

    def sample(self, n: int, seed: int, node_off, nxt, label, backref, key=None, nodes: bool = True, cap: int | None = None):
        """the total weight of every forest of the batch and n derivations of each drawn in proportion to their weight
        (cml_forests_sample): (ln_weight [n_forests, n], n_and [n_forests, n], base [n_forests * n + 1], nodes,
        ln_total [n_forests]); sample (i, r) is nodes[base[i*n+r]:][:n_and[i, r]], in-forest pre-order indices of its AND
        nodes.  key: per forest key of its uniforms (default: the forest's index).  nodes=False asks for weights and sizes
        only (nodes is None).  cap: size of the node buffer handed to the library (default: n * n_nodes, grown once if
        that is too small)."""
        b, keep = self._batch(node_off, nxt, label, backref)
        nf, nn = b.n_forests, int(keep[0][-1])
        lnw, lens = np.empty(max(nf * n, 1)), np.empty(max(nf * n, 1), np.uint32)
        base, total = np.zeros(nf * n + 1, np.uint64), np.empty(max(nf, 1))
        k = None if key is None else _arr(key, np.uint64)
        assert k is None or len(k) == nf

        def call(buf, c):
            return self.lib.cml_forests_sample(self.h, C.byref(b), n, seed, k.ctypes.data_as(_u64p) if k is not None else None,
                                               lnw.ctypes.data_as(_f64p), lens.ctypes.data_as(_u32p), base.ctypes.data_as(_u64p),
                                               buf.ctypes.data_as(_u32p) if buf is not None else None, c,
                                               total.ctypes.data_as(_f64p))
        out = None
        if nodes and n:
            c = n * nn if cap is None else cap
            out = np.empty(max(c, 1), np.uint32)
            rc = call(out, c)
            if rc == -1 and cap is None and int(base[-1]) > c:
                c = int(base[-1])
                out = np.empty(max(c, 1), np.uint32)
                rc = call(out, c)
            self._ok(rc)
            out = out[:int(base[-1])]
        else:
            self._ok(call(None, 0))
        return lnw[:nf * n].reshape(nf, n), lens[:nf * n].reshape(nf, n), base, out, total[:nf]

    def sample_stats(self) -> dict:
        """the last sample() call: scratch bytes of its largest chunk, chunks, kernel time (CUDA events, ms)"""
        return self._decode_stats(self.lib.cml_forests_sample_stats)

    def totals(self):
        v = [C.c_uint64() for _ in range(4)]
        self._ok(self.lib.cml_forests_totals(self.h, *[C.byref(x) for x in v]))
        return dict(zip(("forests", "nodes", "hyperedges", "links"), (x.value for x in v)))

    def estimate(self):
        r = CmlForestEstimateResult()
        self._ok(self.lib.cml_forests_estimate(self.h, C.byref(r)))
        return r.sum_ln_p, r.n_zero, r.n_forests

    def estimate_launch(self):
        self._ok(self.lib.cml_forests_estimate_launch(self.h))

    def estimate_finish(self):
        r = CmlForestEstimateResult()
        self._ok(self.lib.cml_forests_estimate_finish(self.h, C.byref(r)))
        return r.sum_ln_p, r.n_zero, r.n_forests

    def last_time_ms(self):
        ms, nk = C.c_float(), C.c_uint32()
        self._ok(self.lib.cml_forests_last_time_ms(self.h, C.byref(ms), C.byref(nk)))
        return ms.value, nk.value

    def inside(self, n: int) -> np.ndarray:
        v = np.empty(n, np.float64)
        self._ok(self.lib.cml_forests_get_inside(self.h, v.ctypes.data_as(_f64p), n))
        return v

    def counts(self) -> np.ndarray:
        v = np.empty(self.rulespace, np.float64)
        self._ok(self.lib.cml_forests_get_counts(self.h, v.ctypes.data_as(_f64p), self.rulespace))
        return v

    def comm_init_rank(self, n_ranks: int, rank: int, token: bytes):
        assert len(token) == 128
        self._ok(self.lib.cml_forests_comm_init_rank(self.h, n_ranks, rank, token))

    def allreduce_counts(self):
        self._ok(self.lib.cml_forests_allreduce_counts(self.h))

    def reduce_buffer(self):
        p, n = _vp(), C.c_uint64()
        self._ok(self.lib.cml_forests_reduce_buffer(self.h, C.byref(p), C.byref(n)))
        return p.value, n.value

    def maximize(self, prior_total=0.0, add_k=0.0, zero_mode=UNIFORM):
        o = CmlForestNormOpts(prior_total, add_k, zero_mode)
        d, i = C.c_double(), C.c_uint64()
        self._ok(self.lib.cml_forests_maximize(self.h, C.byref(o), C.byref(d), C.byref(i)))
        return d.value, i.value

    def normalize_params(self):
        self._ok(self.lib.cml_forests_normalize_params(self.h))

    def launch_count(self) -> int:
        return int(self.lib.cml_forests_launch_count(self.h))


class ForestJob:
    """A whole forest-em run through the C ABI (what forest-em-b200 does)."""

    def __init__(self, argv: list[str]):
        self.lib = _lib()
        args = [b"forest-em-b200"] + [a.encode() for a in argv]
        arr = (C.c_char_p * len(args))(*args)
        h = _vp()
        rc = self.lib.cml_forest_job_open(C.byref(h), len(args), arr)
        self.h = h
        self._cb = None
        if rc != 0:
            msg = self.lib.cml_forest_job_error(h).decode()
            self.lib.cml_forest_job_close(h)
            self.h = None
            raise CarmelB200Error(rc, msg)

    def _ok(self, rc):
        if rc != 0:
            raise CarmelB200Error(rc, self.lib.cml_forest_job_error(self.h).decode())

    def set_allreduce(self, fn):
        self._cb = ALLREDUCE_FN(lambda user, ptr, n: fn(ptr, n))
        self._ok(self.lib.cml_forest_job_set_allreduce(self.h, self._cb, None))

    def prepare(self):
        self._ok(self.lib.cml_forest_job_prepare(self.h))

    def context(self) -> Forests:
        f = Forests(handle=_vp(self.lib.cml_forest_job_context(self.h)))
        return f

    def train(self):
        self._ok(self.lib.cml_forest_job_train(self.h))

    def write(self):
        self._ok(self.lib.cml_forest_job_write(self.h))

    def stats(self) -> dict:
        i = CmlForestJobInfo()
        self._ok(self.lib.cml_forest_job_stats(self.h, C.byref(i)))
        return {n: getattr(i, n) for n, _ in CmlForestJobInfo._fields_}

    def close(self):
        if self.h:
            self.lib.cml_forest_job_close(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
