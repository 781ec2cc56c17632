"""ctypes binding of the C ABI in include/bppgpu.h (libbppgpu.so).

This is plumbing for tests/, bench.py and __graft_entry__.py: it mirrors the
header one to one (same names, same argument meaning, status codes turned into
``BppGpuError``).  There is no fallback: if the shared library is missing the
import of :func:`lib` raises, and every compute call fails with BPPGPU_E_CUDA
when no sm_100a device is usable.
"""
from __future__ import annotations

import ctypes as C
import os
import pathlib

import numpy as np

PKG_DIR = pathlib.Path(__file__).resolve().parent
LIB_PATH = PKG_DIR / "lib" / "libbppgpu.so"

OK, E_INVALID, E_STATE, E_CUDA, E_NCCL, E_NUMERIC, E_NOMEM = range(7)

MODEL_DIAGONALIZABLE = 1 << 0
MODEL_NONSINGULAR = 1 << 1
MODEL_CLAMP01 = 1 << 2
MODEL_CHR_DERIV = 1 << 3
MODEL_CHR_TAYLOR = 1 << 4
MODEL_EXACT_EXPM = 1 << 5

WANT_P, WANT_DP, WANT_D2P = 1, 2, 4
EVAL_LNL, EVAL_D1, EVAL_D2 = 1, 2, 4

FLAG_KEEP_CLVS = 1 << 0
FLAG_R_SEMANTICS = 1 << 1
FLAG_WEIGHTED_ROOT = 1 << 2
FLAG_NH_DERIV = 1 << 3
FLAG_FORCE_GENERIC = 1 << 4


class BppGpuError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("bppgpu error %d: %s" % (code, msg))
        self.code = code


_dp = C.POINTER(C.c_double)


class ModelDesc(C.Structure):
    _fields_ = [
        ("n_states", C.c_int32),
        ("flags", C.c_uint32),
        ("rate", C.c_double),
        ("right_eigen", _dp),
        ("left_eigen", _dp),
        ("eigen_re", _dp),
        ("eigen_im", _dp),
        ("generator", _dp),
        ("taylor_epsilon", C.c_double),
    ]


class Config(C.Structure):
    _fields_ = [
        ("n_states", C.c_int32),
        ("n_cats", C.c_int32),
        ("n_patterns", C.c_int64),
        ("n_nodes", C.c_int32),
        ("root", C.c_int32),
        ("child_offsets", C.POINTER(C.c_int32)),
        ("children", C.POINTER(C.c_int32)),
        ("n_points", C.c_int32),
        ("n_models", C.c_int32),
        ("n_codes", C.c_int32),
        ("code_bytes", C.c_int32),
        ("code_table", _dp),
        ("device", C.c_int32),
        ("flags", C.c_uint32),
    ]


class Stats(C.Structure):
    _fields_ = [
        ("kernel_launches", C.c_int64),
        ("clv_updates", C.c_int64),
        ("last_eval_ms", C.c_double),
        ("prune_ms", C.c_double),
        ("prune_ms_sum", C.c_double),
        ("prune_count", C.c_int64),
        ("pt_ms_sum", C.c_double),
        ("pt_count", C.c_int64),
        ("hbm_bytes_resident", C.c_int64),
        ("stack_slots", C.c_int32),
        ("path", C.c_int32),
        ("factored_points", C.c_int64),
        ("table_points", C.c_int64),
        ("chr_tiles_tip", C.c_int32),
        ("chr_tiles_dense", C.c_int32),
        ("chr_cblocks_tip", C.c_int32),
        ("chr_cblocks_dense", C.c_int32),
    ]


_lib = None


def lib():
    """The loaded libbppgpu.so (raises if it has not been built: no fallback)."""
    global _lib
    if _lib is None:
        if not LIB_PATH.exists():
            raise ImportError(
                "%s not built; run `python -c 'import __graft_entry__ as g; g.build()'` "
                "(there is no CPU fallback)" % LIB_PATH)
        _lib = C.CDLL(os.fspath(LIB_PATH))
        _lib.bppgpu_last_error.restype = C.c_char_p
    return _lib


def _check(rc):
    if rc != OK:
        raise BppGpuError(rc, lib().bppgpu_last_error().decode())


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def host_model(name, *params):
    """bppgpu_host_model: a named model built by the library's C++ host code (generator + updateMatrices).  Returns a dict with
    Q, V, Vinv, ev (real parts), ev_im, pi (frequencies), flags, rate."""
    pr = _f64(list(params)) if params else np.zeros(0)
    n = C.c_int32(0)
    _check(lib().bppgpu_host_model(name.encode(), pr.ctypes.data_as(_dp), C.c_int32(len(pr)), C.byref(n), None, None,
                                   None, None, None, None, None, None))
    S = n.value
    out = {k: np.zeros((S, S)) for k in ("Q", "V", "Vinv")}
    out.update({k: np.zeros(S) for k in ("ev", "ev_im", "pi")})
    flags, rate = C.c_uint32(0), C.c_double(0)
    _check(lib().bppgpu_host_model(name.encode(), pr.ctypes.data_as(_dp), C.c_int32(len(pr)), C.byref(n), C.byref(flags),
                                   C.byref(rate), *(out[k].ctypes.data_as(_dp) for k in ("Q", "V", "Vinv", "ev", "ev_im", "pi"))))
    out["flags"], out["rate"], out["name"] = flags.value, rate.value, name
    return out


def subtree_patterns(columns, child_off, children, root, leaf_seq):
    """bppgpu_subtree_patterns.  columns: [n_sites][n_seqs] array of fixed-width elements (uint8 / S<k> / uint16 ...).
    Returns (n_patterns[n_nodes], {node: links array} for non-root nodes, root_links, root_weights)."""
    cols = np.ascontiguousarray(columns)
    n_sites, n_seqs = cols.shape
    elem = cols.dtype.itemsize
    child_off = np.ascontiguousarray(child_off, np.int32)
    children = np.ascontiguousarray(children, np.int32)
    leaf_seq = np.ascontiguousarray(leaf_seq, np.int32)
    nn = len(child_off) - 1
    npat = np.zeros(nn, np.int64)
    off = np.zeros(nn + 1, np.int64)
    i64 = C.POINTER(C.c_int64)
    args = (cols.ctypes.data_as(C.POINTER(C.c_uint8)), C.c_int64(n_sites), C.c_int32(n_seqs), C.c_int32(elem), C.c_int32(nn),
            child_off.ctypes.data_as(C.POINTER(C.c_int32)), children.ctypes.data_as(C.POINTER(C.c_int32)), C.c_int32(root),
            leaf_seq.ctypes.data_as(C.POINTER(C.c_int32)), npat.ctypes.data_as(i64), off.ctypes.data_as(i64))
    _check(lib().bppgpu_subtree_patterns(*args, None, None, None))
    links = np.zeros(max(1, int(off[nn])), np.int64)
    rl = np.zeros(max(1, n_sites), np.int64)
    rw = np.zeros(max(1, n_sites), np.uint32)
    _check(lib().bppgpu_subtree_patterns(*args, links.ctypes.data_as(i64), rl.ctypes.data_as(i64),
                                         rw.ctypes.data_as(C.POINTER(C.c_uint32))))
    per = {n: links[off[n]:off[n + 1]].copy() for n in range(nn) if n != root}
    return npat, per, rl[:n_sites], rw[:int(npat[root])]


UNIQUE_ID_BYTES = 128


def comm_unique_id() -> bytes:
    """bppgpu_comm_unique_id: the 128-byte NCCL id rank 0 hands to the other ranks."""
    buf = C.create_string_buffer(UNIQUE_ID_BYTES)
    _check(lib().bppgpu_comm_unique_id(buf))
    return buf.raw


def eval_multi(engines, want=EVAL_LNL):
    """bppgpu_eval_multi: one process, one engine per device over contiguous pattern shards; returns the summed (lnL, d1, d2)."""
    e0 = engines[0]
    arr = (C.c_void_p * len(engines))(*[e._h for e in engines])
    lnl = np.zeros(e0.n_points)
    d1 = np.zeros((e0.n_points, e0.nn)) if want & (EVAL_D1 | EVAL_D2) else None
    d2 = np.zeros((e0.n_points, e0.nn)) if want & EVAL_D2 else None
    _check(lib().bppgpu_eval_multi(arr, C.c_int32(len(engines)), C.c_uint(want), _ptr(lnl), _ptr(d1), _ptr(d2)))
    return lnl, d1, d2


def measure_fp64_peak(device=0):
    """bppgpu_measure_fp64_peak: (DFMA TFLOP/s, DMMA m8n8k4 TFLOP/s) of the device, measured now."""
    a, b = C.c_double(0), C.c_double(0)
    _check(lib().bppgpu_measure_fp64_peak(C.c_int(device), C.byref(a), C.byref(b)))
    return a.value, b.value


def _ptr(a, t=C.c_double):
    return a.ctypes.data_as(C.POINTER(t)) if a is not None else None


def device_count():
    n = C.c_int(0)
    _check(lib().bppgpu_device_count(C.byref(n)))
    return n.value


def site_patterns(columns):
    """bppgpu_site_patterns.  ``columns``: uint8 array [n_sites][col_bytes].  Returns (pattern_site, weights, indices)."""
    cols = np.ascontiguousarray(columns, np.uint8)
    n, w = cols.shape
    ps = np.empty(n, np.int64)
    wt = np.empty(n, np.uint32)
    ix = np.empty(n, np.int64)
    npat = C.c_int64(0)
    _check(lib().bppgpu_site_patterns(cols.ctypes.data_as(C.POINTER(C.c_uint8)), C.c_int64(n), C.c_int32(max(w, 1)),
                                      _ptr(ps, C.c_int64), _ptr(wt, C.c_uint32), _ptr(ix, C.c_int64), C.byref(npat)))
    k = npat.value
    return ps[:k].copy(), wt[:k].copy(), ix


def site_patterns_device(columns, code_bytes=1, tip_codes=True, device=0):
    """bppgpu_site_patterns_device: the same compression on the GPU.  ``columns``: uint8 array [n_sites][col_bytes] (for
    2-byte codes: the little-endian bytes of a uint16 array [n_sites][n_leaves]).  Returns (pattern_site, weights, indices,
    tip codes [n_leaves][n_patterns] or None)."""
    cols = np.ascontiguousarray(columns)
    if cols.dtype == np.uint16:
        code_bytes = 2
        cols = cols.view(np.uint8)
    cols = np.ascontiguousarray(cols, np.uint8)
    n, w = cols.shape
    ps = np.empty(n, np.int64)
    wt = np.empty(n, np.uint32)
    ix = np.empty(n, np.int64)
    tip = np.empty(max(n * w, 1), np.uint8) if tip_codes else None
    npat = C.c_int64(0)
    _check(lib().bppgpu_site_patterns_device(C.c_int(device), cols.ctypes.data_as(C.POINTER(C.c_uint8)), C.c_int64(n),
                                             C.c_int32(max(w, 1)), C.c_int32(code_bytes), _ptr(ps, C.c_int64),
                                             _ptr(wt, C.c_uint32), _ptr(ix, C.c_int64), C.byref(npat),
                                             None if tip is None else tip.ctypes.data_as(C.c_void_p)))
    k = npat.value
    codes = None
    if tip is not None:
        codes = tip[:k * w].view(np.uint8 if code_bytes == 1 else np.uint16).reshape(w // code_bytes, k)   # a view: no second copy
    return ps[:k], wt[:k], ix, codes


def site_patterns_device_raw(columns_ptr, n, col_bytes, ps_ptr, wt_ptr, ix_ptr, tip_ptr=None, code_bytes=1, device=0):
    """bppgpu_site_patterns_device on raw addresses (ints): pinned or device-resident buffers owned by the caller.  Returns the
    number of patterns; the outputs are in the caller's buffers (capacities as in include/bppgpu.h)."""
    npat = C.c_int64(0)
    _check(lib().bppgpu_site_patterns_device(C.c_int(device), C.cast(C.c_void_p(columns_ptr), C.POINTER(C.c_uint8)), C.c_int64(n),
                                             C.c_int32(max(col_bytes, 1)), C.c_int32(code_bytes),
                                             C.cast(C.c_void_p(ps_ptr), C.POINTER(C.c_int64)),
                                             C.cast(C.c_void_p(wt_ptr), C.POINTER(C.c_uint32)),
                                             C.cast(C.c_void_p(ix_ptr), C.POINTER(C.c_int64)), C.byref(npat),
                                             None if tip_ptr is None else C.c_void_p(tip_ptr)))
    return npat.value


class _ModelHolder:
    """Keeps the numpy buffers a ModelDesc points at alive."""

    def __init__(self, S, flags, rate=1.0, V=None, Vinv=None, ev_re=None, ev_im=None, Q=None, eps=1e-4):
        self.arrays = [None if a is None else _f64(a) for a in (V, Vinv, ev_re, ev_im, Q)]
        d = ModelDesc()
        d.n_states = S
        d.flags = flags
        d.rate = rate
        d.right_eigen, d.left_eigen, d.eigen_re, d.eigen_im, d.generator = [_ptr(a) for a in self.arrays]
        d.taylor_epsilon = eps
        self.desc = d


def model_desc(S, flags, **kw):
    return _ModelHolder(S, flags, **kw)


def pt_batch(model: _ModelHolder, t, want=WANT_P, device=0):
    """bppgpu_pt_batch: returns (P, dP, d2P) arrays [n_t][S][S] (None where not wanted)."""
    t = _f64(t).ravel()
    S = model.desc.n_states
    outs = [np.empty((len(t), S, S)) if want & w else None for w in (WANT_P, WANT_DP, WANT_D2P)]
    _check(lib().bppgpu_pt_batch(C.c_int(device), C.byref(model.desc), C.c_int64(len(t)), _ptr(t),
                                 C.c_uint(want), *[_ptr(o) for o in outs]))
    return outs


def _device_address(a):
    """Address of a CUDA tensor or an int address (device memory); None for host arrays."""
    if isinstance(a, int):
        return a
    if hasattr(a, "is_cuda") and a.is_cuda:
        assert a.is_contiguous()
        return a.data_ptr()
    return None


def pairwise_distances(codes, weights, code_table, model: _ModelHolder, freqs, rates, probs, device=0, counts=False,
                       n_leaves=None, n_patterns=None, code_bytes=None):
    """bppgpu_pairwise_distances: ML distance of every pair of tip-code rows (DistanceEstimation::computeMatrix).

    ``codes``: [L][N] uint8 / uint16 numpy array, or device-resident rows (a contiguous CUDA tensor, or an int address of
    device memory with ``n_leaves``, ``n_patterns`` and ``code_bytes`` given) such as site_patterns_device writes.
    ``weights``: [N] (numpy, CUDA tensor or device address).  Returns (dist [L][L], lnl [L][L]) and, with counts=True,
    also the joint code counts [L(L-1)/2][n_codes][n_codes] of the pairs a < b in row-major upper-triangle order."""
    table = _f64(code_table)
    K = table.shape[0]
    addr = _device_address(codes)
    if addr is None:
        c = np.ascontiguousarray(codes)
        if c.dtype not in (np.uint8, np.uint16):
            c = np.ascontiguousarray(c, np.uint8 if K <= 256 else np.uint16)
        L, N = c.shape
        cb = c.dtype.itemsize
        cptr, keep_c = c.ctypes.data_as(C.c_void_p), c
    else:
        if isinstance(codes, int):
            L, N, cb = n_leaves, n_patterns, code_bytes
        else:
            L, N = codes.shape
            cb = codes.element_size()
        cptr, keep_c = C.c_void_p(addr), codes
    waddr = _device_address(weights)
    if waddr is None:
        w = np.ascontiguousarray(weights, np.uint32)
        wptr = _ptr(w, C.c_uint32)
    else:
        w = weights
        wptr = C.cast(C.c_void_p(waddr), C.POINTER(C.c_uint32))
    f, r, p = _f64(freqs), _f64(rates), _f64(probs)
    dist = np.empty((L, L))
    lnl = np.empty((L, L))
    cnt = np.empty((L * (L - 1) // 2, K, K), np.uint32) if counts else None
    _check(lib().bppgpu_pairwise_distances(C.c_int(device), C.byref(model.desc), _ptr(f), C.c_int32(len(r)), _ptr(r), _ptr(p),
                                           C.c_int32(K), C.c_int32(cb), _ptr(table), C.c_int32(L), C.c_int64(N), cptr, wptr,
                                           _ptr(dist), _ptr(lnl), _ptr(cnt, C.c_uint32)))
    del keep_c, w
    return (dist, lnl, cnt) if counts else (dist, lnl)


def pairwise_distances_timing():
    """Device milliseconds of the last pairwise_distances call on this thread: (upload, counts, ML)."""
    v = [C.c_double(0) for _ in range(3)]
    _check(lib().bppgpu_pairwise_distances_timing(*[C.byref(x) for x in v]))
    return tuple(x.value for x in v)


class Engine:
    """Owning wrapper of a ``bppgpu_engine*``."""

    def __init__(self, n_states, n_cats, n_patterns, child_offsets, children, root, code_table,
                 n_points=1, n_models=1, code_bytes=1, device=0, flags=0):
        self._h = C.c_void_p()
        self.child_offsets = np.ascontiguousarray(child_offsets, np.int32)
        self.children = np.ascontiguousarray(children, np.int32)
        self.code_table = _f64(code_table)
        cfg = Config()
        cfg.n_states, cfg.n_cats, cfg.n_patterns = n_states, n_cats, n_patterns
        cfg.n_nodes = len(self.child_offsets) - 1
        cfg.root = root
        cfg.child_offsets = _ptr(self.child_offsets, C.c_int32)
        cfg.children = _ptr(self.children, C.c_int32)
        cfg.n_points, cfg.n_models = n_points, n_models
        cfg.n_codes = self.code_table.shape[0]
        cfg.code_bytes = code_bytes
        cfg.code_table = _ptr(self.code_table)
        cfg.device = device
        cfg.flags = flags
        self.S, self.C, self.N, self.nn = n_states, n_cats, n_patterns, cfg.n_nodes
        self.n_points = n_points
        self.code_bytes = code_bytes
        _check(lib().bppgpu_create(C.byref(cfg), C.byref(self._h)))

    def close(self):
        if self._h:
            lib().bppgpu_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # --- setters ---------------------------------------------------------------
    def leaf_slot(self, node):
        s = C.c_int32(-1)
        _check(lib().bppgpu_leaf_slot(self._h, C.c_int32(node), C.byref(s)))
        return s.value

    def _codes(self, codes):
        return np.ascontiguousarray(codes, np.uint8 if self.code_bytes == 1 else np.uint16)

    def set_tip_codes(self, node, codes):
        a = self._codes(codes)
        _check(lib().bppgpu_set_tip_codes(self._h, C.c_int32(node), a.ctypes.data_as(C.c_void_p)))

    def set_all_tip_codes(self, codes):
        a = self._codes(codes)
        _check(lib().bppgpu_set_all_tip_codes(self._h, a.ctypes.data_as(C.c_void_p)))

    def set_pattern_weights(self, w):
        a = np.ascontiguousarray(w, np.uint32)
        _check(lib().bppgpu_set_pattern_weights(self._h, _ptr(a, C.c_uint32)))

    def set_rates(self, rates, probs):
        r, p = _f64(rates), _f64(probs)
        _check(lib().bppgpu_set_rates(self._h, _ptr(r), _ptr(p)))

    def set_model(self, slot, model: _ModelHolder):
        _check(lib().bppgpu_set_model(self._h, C.c_int32(slot), C.byref(model.desc)))

    def set_models(self, first_slot, models):
        """bppgpu_set_models: a run of slots in one call (pinned staging, one transfer per model)."""
        arr = (ModelDesc * len(models))(*[m.desc for m in models])
        _check(lib().bppgpu_set_models(self._h, C.c_int32(first_slot), C.c_int32(len(models)), arr))

    def set_branch_models(self, point, slots):
        a = np.ascontiguousarray(slots, np.int32)
        _check(lib().bppgpu_set_branch_models(self._h, C.c_int32(point), _ptr(a, C.c_int32)))

    def set_branch_lengths(self, point, t):
        a = _f64(t)
        assert a.size == self.nn
        _check(lib().bppgpu_set_branch_lengths(self._h, C.c_int32(point), _ptr(a)))

    def set_root_freqs(self, point, pi):
        a = _f64(pi)
        _check(lib().bppgpu_set_root_freqs(self._h, C.c_int32(point), _ptr(a)))

    # --- evaluation --------------------------------------------------------------
    def eval(self, want=EVAL_LNL):
        lnl = np.zeros(self.n_points)
        d1 = np.zeros((self.n_points, self.nn)) if want & (EVAL_D1 | EVAL_D2) else None
        d2 = np.zeros((self.n_points, self.nn)) if want & EVAL_D2 else None
        _check(lib().bppgpu_eval(self._h, C.c_uint(want), _ptr(lnl), _ptr(d1), _ptr(d2)))
        return lnl, d1, d2

    def eval_device(self, want, dev_ptr, stream=0):
        _check(lib().bppgpu_eval_device(self._h, C.c_uint(want), C.c_void_p(dev_ptr), C.c_void_p(stream)))

    def eval_status(self):
        """Waits for the last (possibly asynchronous) evaluation; raises BppGpuError(E_NUMERIC) where the reference throws."""
        st = C.c_int32(0)
        _check(lib().bppgpu_eval_status(self._h, C.byref(st)))
        return st.value

    # --- multi-GPU (pattern shards) -------------------------------------------
    def comm_init(self, rank, nranks, unique_id: bytes):
        """Join the NCCL job: from now on eval / eval_device return the whole alignment's lnL, d1, d2 on every rank."""
        assert len(unique_id) == UNIQUE_ID_BYTES
        _check(lib().bppgpu_comm_init(self._h, C.c_int32(rank), C.c_int32(nranks), C.c_char_p(unique_id)))

    def comm_finalize(self):
        _check(lib().bppgpu_comm_finalize(self._h))

    def site_lnl(self, point=0):
        out = np.empty(self.N)
        _check(lib().bppgpu_get_site_lnl(self._h, C.c_int32(point), _ptr(out)))
        return out

    def site_derivatives(self, node, point=0, second=True):
        """bppgpu_get_site_derivatives: ((dL_i/dt)/L_i, (d2L_i/dt2)/L_i) of the branch above `node`, per pattern."""
        a = np.empty(self.N)
        b = np.empty(self.N) if second else None
        _check(lib().bppgpu_get_site_derivatives(self._h, C.c_int32(point), C.c_int32(node), _ptr(a), _ptr(b)))
        return a, b

    def clv(self, node, which=0, point=0):
        out = np.empty((self.N, self.C, self.S))
        ex = np.empty((self.N, self.C), np.int32)
        _check(lib().bppgpu_get_clv(self._h, C.c_int32(point), C.c_int32(node), C.c_int32(which), _ptr(out),
                                    _ptr(ex, C.c_int32)))
        return out, ex

    def node_posteriors(self, node, point=0, full=True):
        """(likelihood at node [N][C][S], its exponents [N][C], posterior probabilities [N][C][S]); full=False asks for
        the posteriors alone (leaves of large problems)."""
        la = np.empty((self.N, self.C, self.S)) if full else None
        ex = np.empty((self.N, self.C), np.int32) if full else None
        post = np.empty((self.N, self.C, self.S))
        _check(lib().bppgpu_get_node_posteriors(self._h, C.c_int32(point), C.c_int32(node), _ptr(la), _ptr(ex, C.c_int32),
                                                _ptr(post)))
        return la, ex, post

    def marginal_posteriors(self, node, point=0, joint=True):
        """MarginalNonRevAncestralStateReconstruction for one node: (posterior [N][S], joint with the father's state
        [N][S][S] indexed [i][node state][father state], or None)."""
        post = np.empty((self.N, self.S))
        jt = np.empty((self.N, self.S, self.S)) if joint else None
        _check(lib().bppgpu_get_marginal_posteriors(self._h, C.c_int32(point), C.c_int32(node), _ptr(post), _ptr(jt)))
        return post, jt

    def ml_ancestral_states(self, point=0):
        """MLAncestralStateReconstruction: (states [n_nodes][N] int32, log joint likelihood of the best assignment [N])"""
        st = np.empty((self.nn, self.N), np.int32)
        best = np.empty(self.N)
        _check(lib().bppgpu_ml_ancestral_states(self._h, C.c_int32(point), _ptr(st, C.c_int32), _ptr(best)))
        return st, best

    def root_reparam_derivatives(self, point=0):
        """(d lnL/d BrLenRoot, d lnL/d RootPosition, d2 lnL/d BrLenRoot^2, d2 lnL/d RootPosition^2) after an eval with D2"""
        out = np.zeros(4)
        _check(lib().bppgpu_get_root_reparam_derivatives(self._h, C.c_int32(point), _ptr(out)))
        return out

    def transition_probabilities(self, node, which=WANT_P, point=0):
        out = np.empty((self.C, self.S, self.S))
        _check(lib().bppgpu_get_transition_probabilities(self._h, C.c_int32(point), C.c_int32(node),
                                                         C.c_uint(which), _ptr(out)))
        return out

    def root_freqs(self, point=0):
        out = np.empty(self.S)
        _check(lib().bppgpu_get_root_freqs(self._h, C.c_int32(point), _ptr(out)))
        return out

    def stats(self):
        s = Stats()
        _check(lib().bppgpu_get_stats(self._h, C.byref(s)))
        out = {k: getattr(s, k) for k, _ in Stats._fields_}
        nf = C.c_int32(0)
        _check(lib().bppgpu_get_frontier_nodes(self._h, C.byref(nf)))
        out["w4c_frontier_nodes"] = nf.value
        return out
