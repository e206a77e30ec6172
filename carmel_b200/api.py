"""ctypes binding of include/carmel_b200.h (the C ABI of the B200-native carmel training path).

This is plumbing for tests, bench.py and the Python driver; the product is the CUDA library.  The
loader fails loudly when libcarmel_b200.so is missing: there is no CPU or PyTorch fallback.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "_build", "libcarmel_b200.so")
CLI_PATH = os.path.join(_HERE, "_build", "carmel-b200")
FOREST_CLI_PATH = os.path.join(_HERE, "_build", "forest-em-b200")

SPACE_LOG, SPACE_SCALED = 0, 1
NO_GROUP = 0xFFFFFFFF
LOCKED_GROUP = 0

OPT_ARC_COUNTS, OPT_NO_ELL, OPT_LANE_MIN, OPT_NO_COUNTS, OPT_NO_FACTOR, OPT_NO_WIDE = 1, 2, 3, 4, 5, 6
OPT_KBEST_SCRATCH_MB, OPT_FREE_BUILD_SCRATCH_MB = 9, 10
OK, ERR_ARG, ERR_CUDA, ERR_STATE, ERR_CYCLE, ERR_NODERIV, ERR_NOT_DENSE = 0, -1, -2, -3, -4, -5, -6

_u32p = C.POINTER(C.c_uint32)
_f64p = C.POINTER(C.c_double)


class CmlModel(C.Structure):
    _fields_ = [
        ("n_arcs", C.c_uint32), ("chain_off", _u32p), ("chain_param", _u32p), ("arc_prior", _f64p),
        ("n_params", C.c_uint32), ("param_group", _u32p), ("param_tie", _u32p), ("n_groups", C.c_uint32),
        ("group_add", _f64p), ("n_ties", C.c_uint32), ("arc_locality_key", C.POINTER(C.c_uint64)),
    ]


class CmlTrellisBatch(C.Structure):
    _fields_ = [
        ("n_ex", C.c_uint64), ("ex_states", _u32p), ("ex_fin", _u32p), ("ex_weight", _f64p),
        ("arc_off", _u32p), ("arc_dst", _u32p), ("arc_id", _u32p),
    ]


class CmlWfstView(C.Structure):
    _fields_ = [("n_states", C.c_uint32), ("final_state", C.c_uint32), ("n_arcs", C.c_uint64),
                ("state_arc_off", _u32p), ("arc_in", _u32p), ("arc_out", _u32p), ("arc_dest", _u32p)]


class CmlStringBatch(C.Structure):
    _fields_ = [("n", C.c_uint64), ("off", C.POINTER(C.c_uint64)), ("sym", _u32p)]


class CmlBuiltTrellises(C.Structure):
    _fields_ = [("batch", CmlTrellisBatch), ("kept_example", _u32p), ("n_dropped", C.c_uint64), ("dropped", _u32p),
                ("pre_arcs", C.c_uint64), ("launches", C.c_uint32), ("peak_states", C.c_uint32),
                ("peak_kept_arcs", C.c_uint32), ("peak_depth", C.c_uint32), ("seconds", C.c_double),
                ("chunks", C.c_uint64), ("kernel_ms", C.c_double), ("owner", C.c_void_p)]


class CmlDenseView(C.Structure):
    _fields_ = [("n_states", C.c_uint32), ("n_symbols", C.c_uint32), ("start", C.c_uint32), ("final_state", C.c_uint32),
                ("arc_src", _u32p), ("arc_dst", _u32p), ("arc_sym", _u32p)]


class CmlSequenceBatch(C.Structure):
    _fields_ = [("n_seq", C.c_uint64), ("seq_off", C.POINTER(C.c_uint64)), ("sym", _u32p), ("seq_weight", _f64p)]


class CmlEstimateResult(C.Structure):
    _fields_ = [("sum_ln_p", C.c_double), ("sum_w_ln_p", C.c_double), ("n_zero", C.c_uint64)]


class CmlGibbsSweepOpts(C.Structure):
    _fields_ = [("mode", C.c_int), ("power", C.c_double), ("seed", C.c_uint64), ("sweep", C.c_uint32),
                ("init_from_params", C.c_int), ("accumulate_dt", C.c_double)]


class CmlJobInfo(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("examples", "trellis_states", "trellis_arcs", "n_params", "n_arcs",
                                          "corpus_pairs", "iterations")] + [("ln_best_ppx", C.c_double),
                                                                            ("last_ln_prob", C.c_double),
                                                                            ("dense", C.c_uint64),
                                                                            ("device_build_s", C.c_double)]


ALLREDUCE_FN = C.CFUNCTYPE(None, C.c_void_p, C.c_void_p, C.c_uint64)


class CarmelB200Error(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"carmel_b200 error {code}: {msg}")
        self.code = code


_lib = None


def load_library(path: str | None = None) -> C.CDLL:
    """Load libcarmel_b200.so (built by carmel_b200/build.py).  Raises if it is missing."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or LIB_PATH
    if not os.path.exists(p):
        raise ImportError(
            f"{p} not found: build it with `python carmel_b200/build.py` (nvcc, sm_100a). "
            "carmel_b200 has no CPU fallback.")
    lib = C.CDLL(p)
    vp = C.c_void_p
    lib.cml_version.restype = C.c_char_p
    lib.cml_create.argtypes = [C.POINTER(vp), C.c_int, C.c_int, C.c_int]
    lib.cml_destroy.argtypes = [vp]
    lib.cml_destroy.restype = None
    lib.cml_last_error.argtypes = [vp]
    lib.cml_last_error.restype = C.c_char_p
    lib.cml_set_stream.argtypes = [vp, vp]
    lib.cml_synchronize.argtypes = [vp]
    lib.cml_launch_count.argtypes = [vp]
    lib.cml_launch_count.restype = C.c_uint64
    lib.cml_set_model.argtypes = [vp, C.POINTER(CmlModel)]
    lib.cml_set_params.argtypes = [vp, _f64p]
    lib.cml_get_params.argtypes = [vp, _f64p]
    lib.cml_snapshot_params.argtypes = [vp, C.c_int]
    lib.cml_restore_params.argtypes = [vp, C.c_int]
    lib.cml_add_trellises.argtypes = [vp, C.POINTER(CmlTrellisBatch)]
    lib.cml_clear_trellises.argtypes = [vp]
    lib.cml_add_sequences.argtypes = [vp, C.POINTER(CmlDenseView), C.POINTER(CmlSequenceBatch)]
    lib.cml_dense_stats.argtypes = [vp, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), _u32p, _u32p]
    lib.cml_dense_kernel.argtypes = [vp, C.POINTER(C.c_int), _u32p, _u32p]
    lib.cml_gibbs_attach_dense.argtypes = [vp, C.POINTER(CmlDenseView), C.POINTER(CmlSequenceBatch)]
    lib.cml_trellis_totals.argtypes = [vp] + [C.POINTER(C.c_uint64)] * 4
    lib.cml_viterbi.argtypes = [vp, _u32p, C.POINTER(C.c_uint64), _u32p, C.c_uint64, _f64p]
    lib.cml_kbest.argtypes = [vp, C.c_uint32, _u32p, C.POINTER(C.c_uint64), _u32p, C.c_uint64, _f64p]
    lib.cml_kbest_stats.argtypes = [vp, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.POINTER(C.c_float)]
    lib.cml_sample.argtypes = [vp, C.c_uint32, C.c_uint64, C.POINTER(C.c_uint64), _u32p, C.POINTER(C.c_uint64), _u32p,
                               C.c_uint64, _f64p, _f64p]
    lib.cml_sample_stats.argtypes = [vp, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.POINTER(C.c_float)]
    lib.cml_build_free_trellises.argtypes = [vp, C.POINTER(CmlWfstView), C.POINTER(CmlStringBatch), C.c_int,
                                             C.POINTER(C.POINTER(CmlBuiltTrellises))]
    lib.cml_free_built_trellises.argtypes = [C.POINTER(CmlBuiltTrellises)]
    lib.cml_free_built_trellises.restype = None
    lib.cml_get_example_layout.argtypes = [vp, C.c_uint64, _u32p, _u32p, _u32p]
    lib.cml_estimate.argtypes = [vp, C.POINTER(CmlEstimateResult)]
    lib.cml_estimate_launch.argtypes = [vp]
    lib.cml_estimate_finish.argtypes = [vp, C.POINTER(CmlEstimateResult)]
    lib.cml_get_example_logprob.argtypes = [vp, _f64p, C.c_uint64]
    lib.cml_get_arc_counts.argtypes = [vp, _f64p]
    lib.cml_reduce_buffer.argtypes = [vp, C.POINTER(vp), C.POINTER(C.c_uint64)]
    lib.cml_use_reduce_buffer.argtypes = [vp, vp, C.c_uint64]
    lib.cml_maximize.argtypes = [vp, C.c_double, _f64p]
    lib.cml_em_step.argtypes = [vp, C.c_double, C.POINTER(CmlEstimateResult), _f64p]
    lib.cml_snapshot_previous.argtypes = [vp, C.c_int]
    lib.cml_comm_unique_id.argtypes = [C.c_char_p]
    lib.cml_comm_init_rank.argtypes = [vp, C.c_int, C.c_int, C.c_char_p]
    lib.cml_comm_init_all.argtypes = [C.POINTER(vp), C.c_int]
    lib.cml_set_comm.argtypes = [vp, vp, C.c_int, C.c_int]
    lib.cml_comm_info.argtypes = [vp, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    lib.cml_allreduce_counts.argtypes = [vp]
    lib.cml_allreduce_buffer.argtypes = [vp, vp, C.c_uint64]
    lib.cml_allreduce_host.argtypes = [vp, _f64p, C.c_uint64]
    lib.cml_collective_count.argtypes = [vp]
    lib.cml_collective_count.restype = C.c_uint64
    lib.cml_job_set_comm.argtypes = [vp, C.c_char_p]
    lib.cml_set_option.argtypes = [vp, C.c_int, C.c_int]
    lib.cml_layout_stats.argtypes = [vp] + [C.POINTER(C.c_uint64)] * 4
    lib.cml_lane_stats.argtypes = [vp] + [C.POINTER(C.c_uint64)] * 4
    lib.cml_wide_stats.argtypes = [vp] + [C.POINTER(C.c_uint64)] * 5
    lib.cml_count_slots.argtypes = [vp]
    lib.cml_count_slots.restype = C.c_uint64
    lib.cml_get_counts.argtypes = [vp, _f64p, C.c_uint64]
    lib.cml_normalize_params.argtypes = [vp]
    lib.cml_last_fb_time_ms.argtypes = [vp, C.POINTER(C.c_float), C.POINTER(C.c_uint32)]
    lib.cml_reduce_buffer_write.argtypes = [vp, _f64p, C.c_uint64]
    lib.cml_reduce_buffer_read.argtypes = [vp, _f64p, C.c_uint64]
    lib.cml_gibbs_sweep.argtypes = [vp, C.POINTER(CmlGibbsSweepOpts)]
    lib.cml_gibbs_sample_capacity.argtypes = [vp]
    lib.cml_gibbs_sample_capacity.restype = C.c_uint64
    lib.cml_gibbs_get_samples.argtypes = [vp, _u32p, _u32p, C.c_uint64]
    lib.cml_job_open.argtypes = [C.POINTER(vp), C.c_int, C.POINTER(C.c_char_p)]
    lib.cml_job_close.argtypes = [vp]
    lib.cml_job_close.restype = None
    lib.cml_job_error.argtypes = [vp]
    lib.cml_job_error.restype = C.c_char_p
    lib.cml_job_set_allreduce.argtypes = [vp, ALLREDUCE_FN, vp]
    lib.cml_job_prepare.argtypes = [vp]
    lib.cml_job_context.argtypes = [vp]
    lib.cml_job_context.restype = vp
    lib.cml_job_train.argtypes = [vp]
    lib.cml_job_write.argtypes = [vp]
    lib.cml_job_stats.argtypes = [vp, C.POINTER(CmlJobInfo)]
    lib.cml_exported_symbols.argtypes = [C.POINTER(C.c_size_t)]
    lib.cml_exported_symbols.restype = C.POINTER(C.c_char_p)
    if path is None:
        _lib = lib
    return lib


def exported_symbols() -> list[str]:
    lib = load_library()
    n = C.c_size_t()
    arr = lib.cml_exported_symbols(C.byref(n))
    return [arr[i].decode() for i in range(n.value)]


def _u32(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.uint32)


def _f64(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.float64)


def _ptr(a: np.ndarray | None, t):
    return a.ctypes.data_as(t) if a is not None else None


class Context:
    """One GPU's training context (cml_ctx).  Mirrors the reference's forward_backward object
    (carmel/src/train.cc:224-460): estimate(), maximize(), save_best / load_best."""

    def __init__(self, device: int = 0, precision: int = 64, space: int = SPACE_LOG):
        self.lib = load_library()
        h = C.c_void_p()
        rc = self.lib.cml_create(C.byref(h), device, precision, space)
        if rc != 0:
            raise CarmelB200Error(rc, self.lib.cml_last_error(None).decode())
        self.h = h
        self.n_arcs = 0
        self.n_params = 0

    def close(self):
        if getattr(self, "h", None):
            self.lib.cml_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int):
        if rc != 0:
            raise CarmelB200Error(rc, self.lib.cml_last_error(self.h).decode())

    def set_stream(self, cuda_stream: int):
        self._check(self.lib.cml_set_stream(self.h, C.c_void_p(cuda_stream)))

    def synchronize(self):
        self._check(self.lib.cml_synchronize(self.h))

    def launch_count(self) -> int:
        return int(self.lib.cml_launch_count(self.h))

    def set_model(self, n_arcs, n_params, param_group, param_tie, n_groups, chain_off=None, chain_param=None,
                  arc_prior=None, group_add=None, n_ties=0):
        keep = []
        m = CmlModel()
        m.n_arcs, m.n_params, m.n_groups, m.n_ties = int(n_arcs), int(n_params), int(n_groups), int(n_ties)

        def u32(a):
            if a is None:
                return None
            a = _u32(a)
            keep.append(a)
            return _ptr(a, _u32p)

        def f64(a):
            if a is None:
                return None
            a = _f64(a)
            keep.append(a)
            return _ptr(a, _f64p)

        m.chain_off, m.chain_param = u32(chain_off), u32(chain_param)
        m.arc_prior, m.group_add = f64(arc_prior), f64(group_add)
        m.param_group, m.param_tie = u32(param_group), u32(param_tie)
        self._check(self.lib.cml_set_model(self.h, C.byref(m)))
        self.n_arcs, self.n_params = int(n_arcs), int(n_params)

    def set_trivial_model(self, n_arcs: int):
        """arc i == parameter i, one joint group, nothing locked (enough for E-step tests)."""
        self.set_model(n_arcs, n_arcs, np.zeros(n_arcs, np.uint32), np.full(n_arcs, NO_GROUP, np.uint32), 1)

    def set_params(self, ln_w):
        a = _f64(ln_w)
        assert a.size == self.n_params
        self._check(self.lib.cml_set_params(self.h, _ptr(a, _f64p)))

    def get_params(self) -> np.ndarray:
        a = np.empty(self.n_params, np.float64)
        self._check(self.lib.cml_get_params(self.h, _ptr(a, _f64p)))
        return a

    def snapshot_params(self, slot: int = 0):
        self._check(self.lib.cml_snapshot_params(self.h, slot))

    def restore_params(self, slot: int = 0):
        self._check(self.lib.cml_restore_params(self.h, slot))

    def add_trellises(self, ex_states, ex_fin, ex_weight, arc_off, arc_dst, arc_id):
        b = CmlTrellisBatch()
        es, ef, ew = _u32(ex_states), _u32(ex_fin), _f64(ex_weight)
        ao, ad, ai = _u32(arc_off), _u32(arc_dst), _u32(arc_id)
        b.n_ex = es.size
        b.ex_states, b.ex_fin, b.ex_weight = _ptr(es, _u32p), _ptr(ef, _u32p), _ptr(ew, _f64p)
        b.arc_off, b.arc_dst, b.arc_id = _ptr(ao, _u32p), _ptr(ad, _u32p), _ptr(ai, _u32p)
        self._check(self.lib.cml_add_trellises(self.h, C.byref(b)))

    def clear_trellises(self):
        self._check(self.lib.cml_clear_trellises(self.h))

    def add_sequences(self, n_states, n_symbols, start, final_state, arc_src, arc_dst, arc_sym, seqs, weights=None):
        """dense-state view (cml_add_sequences): seqs = list of symbol-id sequences.  Raises CarmelB200Error with
        code ERR_NOT_DENSE when the arc table has no transition x emission factorisation."""
        v, b = CmlDenseView(), CmlSequenceBatch()
        a_s, a_d, a_y = _u32(arc_src), _u32(arc_dst), _u32(arc_sym)
        v.n_states, v.n_symbols, v.start, v.final_state = n_states, n_symbols, start, final_state
        v.arc_src, v.arc_dst, v.arc_sym = _ptr(a_s, _u32p), _ptr(a_d, _u32p), _ptr(a_y, _u32p)
        off = np.zeros(len(seqs) + 1, np.uint64)
        off[1:] = np.cumsum([len(q) for q in seqs])
        sym = _u32(np.concatenate([np.asarray(q, np.uint32) for q in seqs]) if len(seqs) else np.zeros(0, np.uint32))
        if sym.size == 0:
            sym = np.zeros(1, np.uint32)
        w = _f64(weights if weights is not None else np.ones(len(seqs)))
        b.n_seq = len(seqs)
        b.seq_off = off.ctypes.data_as(C.POINTER(C.c_uint64))
        b.sym, b.seq_weight = _ptr(sym, _u32p), _ptr(w, _f64p)
        self._check(self.lib.cml_add_sequences(self.h, C.byref(v), C.byref(b)))

    def dense_stats(self) -> dict:
        a, b_ = C.c_uint64(), C.c_uint64()
        c, d = C.c_uint32(), C.c_uint32()
        self._check(self.lib.cml_dense_stats(self.h, C.byref(a), C.byref(b_), C.byref(c), C.byref(d)))
        sp, k, ns = C.c_int(), C.c_uint32(), C.c_uint32()
        self._check(self.lib.cml_dense_kernel(self.h, C.byref(sp), C.byref(k), C.byref(ns)))
        return dict(sequences=int(a.value), positions=int(b_.value), t_slots=int(c.value), e_slots=int(d.value),
                    kernel={1: "sparse", 0: "dense", 2: "dense_tc", -1: None}[int(sp.value)], k=int(k.value), n_states=int(ns.value))

    def trellis_totals(self) -> dict:
        v = [C.c_uint64() for _ in range(4)]
        self._check(self.lib.cml_trellis_totals(self.h, *[C.byref(x) for x in v]))
        return dict(zip(("examples", "states", "arcs", "levels"), (int(x.value) for x in v)))

    # ---- decode (cml_viterbi / cml_kbest) ----
    def _path_arrays(self, n: int, cap: int | None):
        """n_ex, the arc buffer size cap (default: n * total lattice levels) and the zeroed output arrays of n
        derivations per resident lattice: ln_weight, path_len, path_base, path_arcs"""
        t = self.trellis_totals()
        n_ex = t["examples"]
        m = n_ex * n
        if cap is None:
            cap = n * t["levels"]
        return (n_ex, cap, np.zeros(max(m, 1)), np.zeros(max(m, 1), np.uint32), np.zeros(m + 1, np.uint64),
                np.zeros(max(cap, 1), np.uint32))

    def _decode(self, k: int | None, cap: int | None):
        kk = 1 if k is None else k
        n_ex, cap, ln_w, lens, base, arcs = self._path_arrays(kk, cap)
        n = n_ex * kk
        bp = base.ctypes.data_as(C.POINTER(C.c_uint64))
        if k is None:
            rc = self.lib.cml_viterbi(self.h, _ptr(lens, _u32p), bp, _ptr(arcs, _u32p), cap, _ptr(ln_w, _f64p))
        else:
            rc = self.lib.cml_kbest(self.h, k, _ptr(lens, _u32p), bp, _ptr(arcs, _u32p), cap, _ptr(ln_w, _f64p))
        self._check(rc)
        return ln_w[:n].reshape(n_ex, kk), lens[:n].reshape(n_ex, kk), base, arcs

    def kbest(self, k: int, cap: int | None = None):
        """the k best derivations of every resident lattice (cml_kbest): (ln_weight [n_ex, k], path_len [n_ex, k],
        path_base [n_ex * k + 1], path_arcs); derivation (e, r) is path_arcs[path_base[e*k+r]:][:path_len[e, r]].
        cap (default: k * total lattice levels) is the size of the arc buffer handed to the library."""
        return self._decode(int(k), cap)

    def viterbi(self):
        """the best derivation of every resident lattice (cml_viterbi), in kbest()'s shapes with k = 1"""
        return self._decode(None, None)

    def _decode_stats(self, fn) -> dict:
        b, c, ms = C.c_uint64(), C.c_uint64(), C.c_float()
        self._check(fn(self.h, C.byref(b), C.byref(c), C.byref(ms)))
        return {"scratch_bytes": b.value, "chunks": c.value, "kernel_ms": ms.value}

    def kbest_stats(self) -> dict:
        """the last decode call: scratch bytes of its largest chunk, chunks, kernel time (CUDA events, ms)"""
        return self._decode_stats(self.lib.cml_kbest_stats)

    def sample(self, n: int, seed: int, keys=None, cap: int | None = None):
        """the total weight of every resident lattice and n derivations of each drawn in proportion to their weight
        (cml_sample): (ln_total [n_ex], ln_weight [n_ex, n], path_len [n_ex, n], path_base [n_ex * n + 1], path_arcs);
        sample (e, r) is path_arcs[path_base[e*n+r]:][:path_len[e, r]].  keys: the key of each lattice's uniforms
        (default: its index); cap (default: n * total lattice levels) is the size of the arc buffer handed to the
        library.  n = 0 computes ln_total only."""
        n = int(n)
        n_ex, cap, ln_w, lens, base, arcs = self._path_arrays(n, cap)
        m = n_ex * n
        ln_total = np.zeros(max(n_ex, 1))
        kp = None
        if keys is not None:
            keys = np.ascontiguousarray(keys, np.uint64)
            assert keys.size == n_ex, (keys.size, n_ex)
            kp = keys.ctypes.data_as(C.POINTER(C.c_uint64))
        bp = base.ctypes.data_as(C.POINTER(C.c_uint64)) if n else None
        self._check(self.lib.cml_sample(self.h, n, C.c_uint64(int(seed)), kp, _ptr(lens, _u32p) if n else None, bp,
                                        _ptr(arcs, _u32p) if n else None, cap, _ptr(ln_w, _f64p) if n else None,
                                        _ptr(ln_total, _f64p)))
        return ln_total[:n_ex], ln_w[:m].reshape(n_ex, n), lens[:m].reshape(n_ex, n), base, arcs

    def sample_stats(self) -> dict:
        """the last sample() call: scratch bytes of its largest chunk, chunks, kernel time (CUDA events, ms)"""
        return self._decode_stats(self.lib.cml_sample_stats)

    def build_free_trellises(self, wfst: dict, strings, given: int) -> dict:
        """the lattices of the given strings on tape `given` (0 input, 1 output) x the machine, the other tape free
        (cml_build_free_trellises).  wfst: n_states, final_state, state_arc_off, arc_in, arc_out, arc_dest (arc-table
        order, start = state 0); strings: a list of symbol-id sequences, or (off, sym) arrays as the C ABI takes them.
        Returns the batch as numpy arrays (n_ex, ex_states, ex_fin, ex_weight, arc_off, arc_dst, arc_id), kept (string
        index of every lattice), dropped, and the call's statistics; the size of the scratch of one chunk is the option
        OPT_FREE_BUILD_SCRATCH_MB (set_option)."""
        v = CmlWfstView()
        soff, ain, aout, adst = (_u32(wfst[k]) for k in ("state_arc_off", "arc_in", "arc_out", "arc_dest"))
        v.n_states, v.final_state, v.n_arcs = int(wfst["n_states"]), int(wfst["final_state"]), ain.size
        v.state_arc_off, v.arc_in, v.arc_out, v.arc_dest = (_ptr(a, _u32p) for a in (soff, ain, aout, adst))
        if isinstance(strings, tuple):
            off, sym = np.ascontiguousarray(strings[0], np.uint64), _u32(strings[1])
        else:
            off = np.zeros(len(strings) + 1, np.uint64)
            off[1:] = np.cumsum([len(q) for q in strings])
            sym = _u32(np.concatenate([np.asarray(q, np.uint32) for q in strings]) if len(strings) else [])
        sb = CmlStringBatch()
        sb.n = off.size - 1
        sb.off = off.ctypes.data_as(C.POINTER(C.c_uint64))
        sb.sym = _ptr(sym if sym.size else np.zeros(1, np.uint32), _u32p)
        out = C.POINTER(CmlBuiltTrellises)()
        self._check(self.lib.cml_build_free_trellises(self.h, C.byref(v), C.byref(sb), int(given), C.byref(out)))
        try:
            b = out.contents
            t = b.batch
            n_ex = int(t.n_ex)
            ex_states = np.ctypeslib.as_array(t.ex_states, (n_ex,)).copy() if n_ex else np.zeros(0, np.uint32)
            rows = int(ex_states.astype(np.int64).sum()) + n_ex
            take = lambda p, k, dt: np.ctypeslib.as_array(p, (k,)).copy() if k else np.zeros(0, dt)
            arc_off = take(t.arc_off, rows, np.uint32)
            ends = np.cumsum(ex_states.astype(np.int64) + 1) - 1  # each lattice's last row: its arc count
            n_arcs = int(arc_off[ends].astype(np.int64).sum()) if n_ex else 0
            return dict(n_ex=n_ex, ex_states=ex_states, ex_fin=take(t.ex_fin, n_ex, np.uint32),
                        ex_weight=take(t.ex_weight, n_ex, np.float64), arc_off=arc_off,
                        arc_dst=take(t.arc_dst, n_arcs, np.uint32), arc_id=take(t.arc_id, n_arcs, np.uint32),
                        kept=take(b.kept_example, n_ex, np.uint32), dropped=take(b.dropped, int(b.n_dropped), np.uint32),
                        stats=dict(launches=int(b.launches), peak_states=int(b.peak_states),
                                   peak_kept_arcs=int(b.peak_kept_arcs), seconds=float(b.seconds),
                                   chunks=int(b.chunks), kernel_ms=float(b.kernel_ms)))
        finally:
            self.lib.cml_free_built_trellises(out)

    def example_layout(self, e: int, n_states: int):
        nl = C.c_uint32()
        lev = np.empty(n_states, np.uint32)
        loc = np.empty(n_states, np.uint32)
        self._check(self.lib.cml_get_example_layout(self.h, e, C.byref(nl), _ptr(lev, _u32p), _ptr(loc, _u32p)))
        return int(nl.value), lev, loc

    def estimate(self) -> CmlEstimateResult:
        r = CmlEstimateResult()
        self._check(self.lib.cml_estimate(self.h, C.byref(r)))
        return r

    def estimate_launch(self):
        self._check(self.lib.cml_estimate_launch(self.h))

    def em_step(self, rate: float = 1.0):
        """one whole EM iteration (E-step, all-reduce when a communicator is set, M-step), one host synchronisation;
        returns (CmlEstimateResult of the weights the iteration started from, max weight change)"""
        r = CmlEstimateResult()
        d = C.c_double()
        self._check(self.lib.cml_em_step(self.h, rate, C.byref(r), C.cast(C.byref(d), _f64p)))
        return r, float(d.value)

    def snapshot_previous(self, slot: int = 0):
        self._check(self.lib.cml_snapshot_previous(self.h, slot))

    def comm_init_rank(self, n_ranks: int, rank: int, token: bytes):
        assert len(token) == 128
        self._check(self.lib.cml_comm_init_rank(self.h, n_ranks, rank, token))

    def allreduce_counts(self):
        self._check(self.lib.cml_allreduce_counts(self.h))

    def collective_count(self) -> int:
        return int(self.lib.cml_collective_count(self.h))

    def estimate_finish(self) -> CmlEstimateResult:
        r = CmlEstimateResult()
        self._check(self.lib.cml_estimate_finish(self.h, C.byref(r)))
        return r

    def example_logprob(self, n: int) -> np.ndarray:
        a = np.empty(n, np.float64)
        self._check(self.lib.cml_get_example_logprob(self.h, _ptr(a, _f64p), n))
        return a

    def set_option(self, option: int, value: int):
        self._check(self.lib.cml_set_option(self.h, option, value))

    def layout_stats(self) -> dict:
        v = [C.c_uint64() for _ in range(4)]
        self._check(self.lib.cml_layout_stats(self.h, *[C.byref(x) for x in v]))
        return dict(zip(("ell_examples", "ell_arcs", "ell_records", "csr_examples"), (int(x.value) for x in v)))

    def lane_stats(self) -> dict:
        v = [C.c_uint64() for _ in range(4)]
        self._check(self.lib.cml_lane_stats(self.h, *[C.byref(x) for x in v]))
        return dict(zip(("lane_examples", "lane_arcs", "lane_records", "tiles"), (int(x.value) for x in v)))

    def wide_stats(self) -> dict:
        v = [C.c_uint64() for _ in range(5)]
        self._check(self.lib.cml_wide_stats(self.h, *[C.byref(x) for x in v]))
        return dict(zip(("wide_examples", "wide_arcs", "wide_records", "arc_classes", "state_classes"),
                        (int(x.value) for x in v)))

    def count_slots(self) -> int:
        return int(self.lib.cml_count_slots(self.h))

    def counts(self) -> np.ndarray:
        a = np.empty(self.count_slots(), np.float64)
        self._check(self.lib.cml_get_counts(self.h, _ptr(a, _f64p), a.size))
        return a

    def get_counts_ptr(self, host_ptr: int, n: int):
        self._check(self.lib.cml_get_counts(self.h, C.cast(C.c_void_p(host_ptr), _f64p), n))

    def arc_counts(self) -> np.ndarray:
        a = np.empty(self.n_arcs, np.float64)
        self._check(self.lib.cml_get_arc_counts(self.h, _ptr(a, _f64p)))
        return a

    def reduce_buffer(self) -> tuple[int, int]:
        p = C.c_void_p()
        n = C.c_uint64()
        self._check(self.lib.cml_reduce_buffer(self.h, C.byref(p), C.byref(n)))
        return int(p.value), int(n.value)

    def use_reduce_buffer(self, device_ptr: int | None, n_doubles: int = 0):
        self._check(self.lib.cml_use_reduce_buffer(self.h, C.c_void_p(device_ptr or 0), n_doubles))

    def last_fb_time_ms(self) -> tuple[float, int]:
        ms = C.c_float()
        nk = C.c_uint32()
        self._check(self.lib.cml_last_fb_time_ms(self.h, C.byref(ms), C.byref(nk)))
        return float(ms.value), int(nk.value)

    def set_params_ptr(self, host_ptr: int):
        """cml_set_params from a raw (e.g. pinned) host pointer"""
        self._check(self.lib.cml_set_params(self.h, C.cast(C.c_void_p(host_ptr), _f64p)))

    def get_params_ptr(self, host_ptr: int):
        self._check(self.lib.cml_get_params(self.h, C.cast(C.c_void_p(host_ptr), _f64p)))

    def get_arc_counts_ptr(self, host_ptr: int):
        self._check(self.lib.cml_get_arc_counts(self.h, C.cast(C.c_void_p(host_ptr), _f64p)))

    def maximize(self, rate: float = 1.0) -> float:
        d = C.c_double()
        self._check(self.lib.cml_maximize(self.h, rate, C.byref(d)))
        return float(d.value)

    def normalize_params(self):
        self._check(self.lib.cml_normalize_params(self.h))

    # ---- --crp Gibbs sampling (cml_gibbs_*) ----
    def gibbs_sweep(self, mode: int, sweep: int, seed: int = 1, power: float = 1.0, accumulate_dt: float = 0.0,
                    init_from_params: bool = False):
        """one sweep over all blocks; mode 0 = sequential (exact collapsed sampler), 1 = batched"""
        o = CmlGibbsSweepOpts(mode, power, seed, sweep, int(init_from_params), accumulate_dt)
        self._check(self.lib.cml_gibbs_sweep(self.h, C.byref(o)))

    def gibbs_sample_capacity(self) -> int:
        return int(self.lib.cml_gibbs_sample_capacity(self.h))

    def gibbs_get_samples_ptr(self, len_ptr: int, arcs_ptr: int, cap: int):
        self._check(self.lib.cml_gibbs_get_samples(self.h, C.cast(len_ptr, _u32p), C.cast(arcs_ptr, _u32p), cap))


def comm_unique_id() -> bytes:
    """128-byte NCCL rendezvous token (cml_comm_unique_id): create on rank 0, broadcast to the other ranks"""
    buf = C.create_string_buffer(128)
    rc = load_library().cml_comm_unique_id(buf)
    if rc != 0:
        raise CarmelB200Error(rc, "cml_comm_unique_id failed (libnccl.so.2 not loadable?)")
    return buf.raw


class Job:
    """One `carmel -t ...` run (cml_job): argv in carmel's grammar.  After prepare() the job's Context
    (borrowed, owned by the job) can be driven step by step; train() runs the reference's EM loop."""

    def __init__(self, argv: list[str], allreduce=None, comm_token: bytes | None = None):
        self.lib = load_library()
        args = ["carmel-b200", *argv]
        arr = (C.c_char_p * len(args))(*[a.encode() for a in args])
        h = C.c_void_p()
        rc = self.lib.cml_job_open(C.byref(h), len(args), arr)
        self.h = h
        if rc != 0:
            msg = self.lib.cml_job_error(h).decode()
            self.close()
            raise CarmelB200Error(rc, msg)
        self._cb = None
        if allreduce is not None:
            self._cb = ALLREDUCE_FN(lambda user, ptr, n: allreduce(int(ptr), int(n)))
            self.lib.cml_job_set_allreduce(self.h, self._cb, None)
        if comm_token is not None:  # NCCL rendezvous token (comm_unique_id on rank 0, shipped to every rank)
            assert len(comm_token) == 128
            self._check(self.lib.cml_job_set_comm(self.h, comm_token))
        self.ctx = None

    def _check(self, rc):
        if rc != 0:
            raise CarmelB200Error(rc, self.lib.cml_job_error(self.h).decode())

    def prepare(self) -> "Context":
        self._check(self.lib.cml_job_prepare(self.h))
        ctx = Context.__new__(Context)
        ctx.lib = self.lib
        ctx.h = None  # borrowed: never destroyed from Python
        ctx._borrowed = C.c_void_p(self.lib.cml_job_context(self.h))
        info = self.stats()
        ctx.n_arcs, ctx.n_params = info["n_arcs"], info["n_params"]
        ctx.h = ctx._borrowed
        ctx.close = lambda: None
        self.ctx = ctx
        return ctx

    def stats(self) -> dict:
        i = CmlJobInfo()
        self._check(self.lib.cml_job_stats(self.h, C.byref(i)))
        return {n: getattr(i, n) for n, _ in CmlJobInfo._fields_}

    def train(self):
        self._check(self.lib.cml_job_train(self.h))

    def write(self):
        self._check(self.lib.cml_job_write(self.h))

    def close(self):
        if getattr(self, "h", None):
            self.lib.cml_job_close(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
