"""wfsa_b200 -- ctypes glue over libwfsa_b200.so (C ABI: include/wfsa_dev.h, include/wfsa_host.h).

Python is plumbing here (tests, bench.py): the product is the shared library.  Loading fails
loudly when the library has not been built (``make -C w-fsa_b200``); nothing in this package
computes on the CPU.
"""
import ctypes as C
import json
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
PKG_ROOT = os.path.abspath(os.path.join(_HERE, "..", ".."))
LIB_PATH = os.path.join(PKG_ROOT, "_build", "libwfsa_b200.so")
UNIQUE_ID_BYTES = 128

DEV_SYMBOLS = [
    "wfsa_dev_create", "wfsa_dev_structure", "wfsa_dev_set_param_map", "wfsa_dev_eval", "wfsa_dev_upload_x",
    "wfsa_dev_eval_launch", "wfsa_dev_eval_fetch", "wfsa_dev_sync", "wfsa_dev_set_path_blocks", "wfsa_dev_hessian",
    "wfsa_dev_viterbi", "wfsa_dev_viterbi_paths", "wfsa_dev_nbest", "wfsa_dev_sample",
    "wfsa_dev_comm_unique_id", "wfsa_dev_comm_init", "wfsa_dev_allreduce_f64", "wfsa_dev_timer_begin", "wfsa_dev_timer_begin_steps",
    "wfsa_dev_timer_end", "wfsa_dev_timer_kernel_ms", "wfsa_dev_timer_split_ms", "wfsa_dev_timer_step_ms", "wfsa_dev_timer_phase_ms", "wfsa_dev_eval6_phases", "wfsa_dev_l2_flush", "wfsa_dev_rank_barrier", "wfsa_dev_get_info", "wfsa_dev_destroy", "wfsa_dev_held_bytes", "wfsa_dev_last_error",
    "wfsa_dev_version", "wfsa_lattice_compile", "wfsa_segmented_compile", "wfsa_segmented_get",
    "wfsa_segmented_free",
]
HOST_SYMBOLS = [
    "wfsa_host_parse", "wfsa_host_last_error", "wfsa_host_kkt_solve", "wfsa_philox4x32_10", "wfsa_session_create", "wfsa_session_destroy", "wfsa_session_error",
    "wfsa_session_describe", "wfsa_session_n", "wfsa_session_k", "wfsa_session_n_recognised_local", "wfsa_session_init",
    "wfsa_session_eval", "wfsa_session_hessian", "wfsa_session_step", "wfsa_session_halt", "wfsa_session_get_x",
    "wfsa_session_renormalize", "wfsa_session_result", "wfsa_session_dump", "wfsa_session_backend",
]

I32P = C.POINTER(C.c_int32)
I64P = C.POINTER(C.c_int64)
U32P = C.POINTER(C.c_uint32)
F64P = C.POINTER(C.c_double)
U8P = C.POINTER(C.c_uint8)


class FsaDesc(C.Structure):
    _fields_ = [("n_states", C.c_int32), ("start_state", C.c_int32), ("end_state", C.c_int32), ("n_symbols", C.c_int32),
                ("n_raw_params", C.c_int32), ("emis_row", I32P), ("emis_tok_off", I32P), ("emis_tok", I32P),
                ("emis_param", I32P), ("trans_row", I32P), ("trans_dst", I32P), ("trans_param", I32P)]


class CorpusDesc(C.Structure):
    _fields_ = [("n_strings", C.c_int64), ("offsets", I64P), ("tokens", I32P), ("p", F64P)]


class DevOptions(C.Structure):
    _fields_ = [("device", C.c_int32), ("force_kernel", C.c_int32), ("accum_mode", C.c_int32), ("reserved", C.c_int32)]


class DevInfo(C.Structure):
    _fields_ = [("kernel", C.c_int32), ("accum_mode", C.c_int32), ("n_trans", C.c_int32), ("n_emis", C.c_int32),
                ("n_arcs", C.c_int32), ("n_slots", C.c_int32), ("max_candidates", C.c_int32), ("sm_count", C.c_int32),
                ("grid", C.c_int32), ("block", C.c_int32), ("n_strings", C.c_int64), ("n_active_strings", C.c_int64),
                ("n_tokens", C.c_int64), ("n_active_tokens", C.c_int64), ("smem_bytes", C.c_int64),
                ("table_bytes", C.c_int64), ("kernels_launched", C.c_int64), ("fixed_point_scale_log2", C.c_double),
                ("lattice_words", C.c_int64), ("lattice_edges", C.c_int64), ("lattice_bridge_edges", C.c_int64),
                ("n_overflow_strings", C.c_int64), ("pool_slots", C.c_int32), ("eval_path", C.c_int32),
                ("seg_types", C.c_int64), ("seg_region_instances", C.c_int64), ("seg_region_edges", C.c_int64),
                ("seg_type_edges", C.c_int64), ("seg_host_ms", C.c_double), ("e6_big_groups", C.c_int64),
                ("e6_big_dedicate", C.c_int32), ("e6_big_slots", C.c_int32), ("e6_big_rows", C.c_int32),
                ("e6_max_big_rows", C.c_int32), ("e6_two_warp_eligible", C.c_int32)]


class PathBlocks(C.Structure):
    _fields_ = [("n_blocks", C.c_int64), ("path_off", I64P), ("col_off", I64P), ("cols", I32P), ("val_off", I64P),
                ("counts", F64P), ("p", F64P)]


class SessionOptions(C.Structure):
    _fields_ = [("device", C.c_int32), ("force_kernel", C.c_int32), ("accum_mode", C.c_int32), ("accum_variant", C.c_int32),
                ("rank", C.c_int32), ("nranks", C.c_int32), ("unique_id", C.c_void_p)]


class WfsaError(RuntimeError):
    def __init__(self, code, message):
        super().__init__("wfsa error %d: %s" % (code, message))
        self.code = code
        self.message = message


_lib = None


def lib():
    """The shared library; raises if it has not been built -- there is no fallback."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError("%s is missing: build it with `make -C w-fsa_b200` (or __graft_entry__.build())" % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        L.wfsa_dev_last_error.restype = C.c_char_p
        L.wfsa_dev_last_error.argtypes = [C.c_void_p]
        L.wfsa_dev_version.restype = C.c_char_p
        L.wfsa_host_last_error.restype = C.c_char_p
        L.wfsa_session_error.restype = C.c_char_p
        L.wfsa_session_error.argtypes = [C.c_void_p]
        L.wfsa_session_describe.restype = C.c_char_p
        L.wfsa_session_describe.argtypes = [C.c_void_p]
        L.wfsa_session_dump.restype = C.c_char_p
        L.wfsa_session_dump.argtypes = [C.c_void_p, C.c_int]
        L.wfsa_session_backend.restype = C.c_void_p
        L.wfsa_session_backend.argtypes = [C.c_void_p]
        for name in ("wfsa_session_n", "wfsa_session_k", "wfsa_session_n_recognised_local"):
            getattr(L, name).argtypes = [C.c_void_p]
        L.wfsa_session_destroy.argtypes = [C.c_void_p]
        L.wfsa_session_destroy.restype = None
        L.wfsa_dev_destroy.argtypes = [C.c_void_p]
        L.wfsa_dev_destroy.restype = None
        L.wfsa_dev_held_bytes.argtypes = []
        L.wfsa_dev_held_bytes.restype = C.c_int64
        L.wfsa_session_create.argtypes = [C.c_char_p, C.c_size_t, C.c_char_p, C.c_size_t, C.c_char_p,
                                          C.POINTER(SessionOptions), C.POINTER(C.c_void_p)]
        L.wfsa_host_parse.argtypes = [C.c_char_p, C.c_size_t, C.c_char_p, C.c_size_t, C.POINTER(C.c_char_p)]
        L.wfsa_session_init.argtypes = [C.c_void_p, C.c_int, F64P]
        L.wfsa_session_eval.argtypes = [C.c_void_p, F64P, F64P, F64P, F64P, F64P]
        L.wfsa_session_hessian.argtypes = [C.c_void_p, F64P, F64P]
        L.wfsa_session_step.argtypes = [C.c_void_p, C.c_double, F64P, C.POINTER(C.c_int)]
        L.wfsa_session_halt.argtypes = [C.c_void_p, C.c_double, C.POINTER(C.c_int)]
        L.wfsa_session_get_x.argtypes = [C.c_void_p, F64P, C.c_int]
        L.wfsa_session_renormalize.argtypes = [C.c_void_p]
        L.wfsa_session_result.argtypes = [C.c_void_p, F64P]
        L.wfsa_dev_create.argtypes = [C.POINTER(FsaDesc), C.POINTER(CorpusDesc), C.POINTER(DevOptions), C.POINTER(C.c_void_p)]
        L.wfsa_dev_structure.argtypes = [C.c_void_p, U8P, F64P, U8P]
        L.wfsa_dev_set_param_map.argtypes = [C.c_void_p, I32P, C.c_int32, U8P]
        L.wfsa_dev_eval.argtypes = [C.c_void_p, C.c_void_p, F64P, C.c_void_p, C.c_void_p]     # raw addresses: cheaper to marshal per call
        L.wfsa_dev_upload_x.argtypes = [C.c_void_p, F64P]
        L.wfsa_dev_eval_launch.argtypes = [C.c_void_p]
        L.wfsa_dev_eval_fetch.argtypes = [C.c_void_p, F64P, F64P, F64P]
        L.wfsa_dev_sync.argtypes = [C.c_void_p]
        L.wfsa_dev_set_path_blocks.argtypes = [C.c_void_p, C.POINTER(PathBlocks)]
        L.wfsa_dev_hessian.argtypes = [C.c_void_p, F64P, F64P, F64P]
        L.wfsa_dev_viterbi.argtypes = [C.c_void_p, F64P, F64P, I64P]
        L.wfsa_dev_viterbi_paths.argtypes = [C.c_void_p, I32P, I32P]
        L.wfsa_dev_nbest.argtypes = [C.c_void_p, F64P, C.c_int32, F64P, I64P]
        L.wfsa_dev_sample.argtypes = [C.c_void_p, F64P, C.c_int32, C.c_uint64, F64P, F64P, I64P]
        L.wfsa_philox4x32_10.argtypes = [U32P, U32P, U32P]
        L.wfsa_philox4x32_10.restype = None
        L.wfsa_dev_comm_unique_id.argtypes = [C.c_void_p]
        L.wfsa_dev_comm_init.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int]
        L.wfsa_dev_allreduce_f64.argtypes = [C.c_void_p, F64P, C.c_int, C.c_int]
        L.wfsa_dev_timer_begin.argtypes = [C.c_void_p]
        L.wfsa_dev_timer_end.argtypes = [C.c_void_p, C.POINTER(C.c_float)]
        L.wfsa_dev_timer_kernel_ms.argtypes = [C.c_void_p, C.POINTER(C.c_float), I64P]
        L.wfsa_dev_timer_split_ms.argtypes = [C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_float)]
        L.wfsa_dev_timer_step_ms.argtypes = [C.c_void_p, C.POINTER(C.c_float), I64P]
        L.wfsa_dev_l2_flush.argtypes = [C.c_void_p]
        L.wfsa_dev_rank_barrier.argtypes = [C.c_void_p]
        L.wfsa_dev_timer_phase_ms.argtypes = [C.c_void_p, C.POINTER(C.c_float)]
        L.wfsa_dev_eval6_phases.argtypes = [C.c_void_p, F64P, C.c_int]
        L.wfsa_dev_get_info.argtypes = [C.c_void_p, C.POINTER(DevInfo)]
        L.wfsa_lattice_compile.argtypes = [C.POINTER(FsaDesc), I32P, I32P, C.c_int32, C.c_int32, C.POINTER(C.c_uint32), C.c_int64,
                                           I64P, I32P, I32P, C.c_int32, I32P]
        L.wfsa_segmented_compile.argtypes = [C.POINTER(FsaDesc), C.POINTER(CorpusDesc), I32P, C.c_int32, C.c_double,
                                             C.POINTER(C.c_void_p)]
        L.wfsa_segmented_get.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_void_p), I64P]
        L.wfsa_segmented_free.argtypes = [C.c_void_p]
        L.wfsa_segmented_free.restype = None
        _lib = L
    return _lib


_SEG_ARRAYS = [("rwords", np.uint32), ("rgoff", np.int64), ("rgrows", np.int32), ("typeW", np.float64), ("swords", np.uint32),
               ("sgoff", np.int64), ("sgref", np.int32), ("ksid", np.int32), ("kp", np.float64), ("overflow", np.int32),
               ("rejected", np.int32), ("const_acc", np.int64), ("stats", np.int64), ("hb_path_off", np.int64), ("hb_col_off", np.int64), ("hb_val_off", np.int64),
               ("hb_cols", np.int32), ("hb_counts", np.float64), ("hb_p", np.float64), ("hb_slot", np.int32), ("pwords", np.uint32),
               ("pgoff", np.int64)]


def segmented_compile(lowered, trimmed=None, n_slots=16, fx_scale=1.0):
    """Host-only: the segmented compiled form of a shard (include/wfsa_dev.h wfsa_segmented_*) as numpy arrays,
    plus the combined-arc table (arc -> transition edge, emission edge or -1)."""
    L = lib()
    fd, cd = lowered.fsa_desc(), lowered.corpus_desc()
    tr = None if trimmed is None else np.ascontiguousarray(trimmed, dtype=np.int32)
    h = C.c_void_p()
    rc = L.wfsa_segmented_compile(C.byref(fd), C.byref(cd), _p(tr, I32P), n_slots, fx_scale, C.byref(h))
    if rc != 0:
        raise WfsaError(rc, L.wfsa_dev_last_error(None).decode())
    out = {}
    try:
        for i, (name, dt) in enumerate(_SEG_ARRAYS):
            ptr, cnt = C.c_void_p(), C.c_int64()
            L.wfsa_segmented_get(h, i, C.byref(ptr), C.byref(cnt))
            if cnt.value:
                buf = (C.c_char * (cnt.value * np.dtype(dt).itemsize)).from_address(ptr.value)
                out[name] = np.frombuffer(buf, dtype=dt).copy()
            else:
                out[name] = np.zeros(0, dtype=dt)
    finally:
        L.wfsa_segmented_free(h)
    return out


def _p(a, t):
    return None if a is None else a.ctypes.data_as(t)


def _jfloat(v):
    return float(v) if isinstance(v, str) else v


def parse(fsa_text, corpus_text):
    """Parse both files on the host (no device); returns the JSON description as a dict."""
    L = lib()
    fa = fsa_text.encode("latin-1") if isinstance(fsa_text, str) else fsa_text
    co = corpus_text.encode("latin-1") if isinstance(corpus_text, str) else corpus_text
    out = C.c_char_p()
    rc = L.wfsa_host_parse(fa, len(fa), co, len(co), C.byref(out))
    if rc != 0:
        raise WfsaError(rc, L.wfsa_host_last_error().decode("latin-1"))
    return json.loads(out.value.decode("latin-1"))


class Lowered:
    """Index-based descriptors (include/wfsa_dev.h) built in Python from a parse() description.
    Edge ids: transitions in state order, then emissions in state order."""

    def __init__(self, desc, corpus=None, normalise=True):
        names = desc["state_names"]
        sid = {n: i for i, n in enumerate(names)}
        self.desc = desc
        self.n_states, self.start, self.end = len(names), desc["start"], desc["end"]
        emis = [[] for _ in names]
        trans = [[] for _ in names]
        for e in desc["edges"]:
            (emis if e["kind"] == "E" else trans)[sid[e["state"]]].append(e)
        sym = {}
        for es in emis:
            for e in es:
                for ch in e["label"].encode("latin-1"):
                    sym.setdefault(ch, len(sym))
        self.sym = sym
        self.n_symbols = len(sym)
        self.n_raw = desc["raw_parameters"]
        emis_row, tok_off, tok, eparam, trow, tdst, tparam = [0], [0], [], [], [0], [], []
        self.trans_edges, self.emis_edges = [], []
        for s in range(len(names)):
            for e in emis[s]:
                tok.extend(sym[ch] for ch in e["label"].encode("latin-1"))
                tok_off.append(len(tok))
                eparam.append(e["raw"])
                self.emis_edges.append(e)
            emis_row.append(len(eparam))
            for t in trans[s]:
                tdst.append(sid[t["label"]])
                tparam.append(t["raw"])
                self.trans_edges.append(t)
            trow.append(len(tdst))
        i32 = lambda v: np.ascontiguousarray(np.array(v, dtype=np.int32).reshape(-1))
        self.emis_row, self.emis_tok_off, self.emis_tok, self.emis_param = i32(emis_row), i32(tok_off), i32(tok), i32(eparam)
        self.trans_row, self.trans_dst, self.trans_param = i32(trow), i32(tdst), i32(tparam)
        self.n_trans, self.n_emis = len(tdst), len(eparam)
        self.edges = self.trans_edges + self.emis_edges
        if corpus is None:
            corpus = [(w["word"], _jfloat(w["weight"])) for w in desc.get("corpus", [])]
        self.set_corpus(corpus, normalise)

    def set_corpus(self, corpus, normalise=True):
        offs, toks = [0], []
        for w, _ in corpus:
            b = w.encode("latin-1") if isinstance(w, str) else w
            toks.extend(self.sym.get(ch, -1) for ch in b)
            offs.append(len(toks))
        self.offsets = np.array(offs, dtype=np.int64)
        self.tokens = np.ascontiguousarray(np.array(toks, dtype=np.int32).reshape(-1))
        wts = np.array([c for _, c in corpus], dtype=np.float64)
        self.p = wts / wts.sum() if (normalise and len(wts)) else wts
        self.words = [w for w, _ in corpus]

    def set_tokens(self, offsets, tokens, p):
        self.offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        self.tokens = np.ascontiguousarray(tokens, dtype=np.int32)
        self.p = np.ascontiguousarray(p, dtype=np.float64)
        self.words = None

    def fsa_desc(self):
        d = FsaDesc()
        d.n_states, d.start_state, d.end_state = self.n_states, self.start, self.end
        d.n_symbols, d.n_raw_params = self.n_symbols, self.n_raw
        for k in ("emis_row", "emis_tok_off", "emis_tok", "emis_param", "trans_row", "trans_dst", "trans_param"):
            setattr(d, k, _p(getattr(self, k), I32P))
        return d

    def corpus_desc(self, first=0, count=None):
        n = len(self.offsets) - 1
        count = n - first if count is None else count
        offs = np.ascontiguousarray(self.offsets[first:first + count + 1] - self.offsets[first])
        toks = np.ascontiguousarray(self.tokens[self.offsets[first]:self.offsets[first + count]])
        p = np.ascontiguousarray(self.p[first:first + count])
        d = CorpusDesc()
        d.n_strings = count
        d.offsets, d.tokens, d.p = _p(offs, I64P), _p(toks, I32P), _p(p, F64P)
        d._keep = (offs, toks, p)
        return d

    def edge_logweights(self, x, trimmed):
        """log-weight of every edge (transitions then emissions) for trimmed-parameter vector x."""
        out = np.zeros(self.n_trans + self.n_emis)
        params = np.concatenate([self.trans_param, self.emis_param])
        for i, r in enumerate(params):
            if r < 0:
                continue
            t = trimmed[r]
            out[i] = -np.inf if t == -2 else (0.0 if t == -1 else x[t])
        return out[:self.n_trans].copy(), out[self.n_trans:].copy()


class Device:
    """Thin wrapper over the wfsa_dev_* C ABI."""

    def __init__(self, lowered, device=0, force_kernel=0, accum_mode=0, accum_variant=0, first=0, count=None):
        self.L = lib()
        self.low = lowered
        self.h = C.c_void_p()
        fd = lowered.fsa_desc()
        self._cd = lowered.corpus_desc(first, count)
        self.n_strings = int(self._cd.n_strings)
        opt = DevOptions(device, force_kernel, accum_mode, accum_variant)
        rc = self.L.wfsa_dev_create(C.byref(fd), C.byref(self._cd), C.byref(opt), C.byref(self.h))
        if rc != 0:
            raise WfsaError(rc, self.L.wfsa_dev_last_error(None).decode())
        self.n = None

    def _ck(self, rc):
        if rc != 0:
            raise WfsaError(rc, self.L.wfsa_dev_last_error(self.h).decode())

    def comm_init(self, uid, rank, nranks):
        self._uid = C.create_string_buffer(bytes(uid), UNIQUE_ID_BYTES)
        self._ck(self.L.wfsa_dev_comm_init(self.h, self._uid, rank, nranks))

    def structure(self):
        rec = np.zeros(self.n_strings, dtype=np.uint8)
        pc = np.zeros(self.n_strings, dtype=np.float64)
        used = np.zeros(max(self.low.n_raw, 1), dtype=np.uint8)
        self._ck(self.L.wfsa_dev_structure(self.h, _p(rec, U8P), _p(pc, F64P), _p(used, U8P)))
        return rec, pc, used[:self.low.n_raw]

    def set_param_map(self, trimmed, n, recognised=None):
        t = np.ascontiguousarray(trimmed, dtype=np.int32)
        r = None if recognised is None else np.ascontiguousarray(recognised, dtype=np.uint8)
        self._ck(self.L.wfsa_dev_set_param_map(self.h, _p(t, I32P), n, _p(r, U8P)))
        self.n = n

    def eval(self, x, want_logq=True):
        if not (isinstance(x, np.ndarray) and x.dtype == np.float64 and x.flags.c_contiguous):
            x = np.ascontiguousarray(x, dtype=np.float64)
        ll = C.c_double()
        grad = np.empty(max(self.n, 1))
        logq = np.zeros(max(self.n_strings, 1)) if want_logq else None
        self._ck(self.L.wfsa_dev_eval(self.h, x.ctypes.data, C.byref(ll), logq.ctypes.data if want_logq else None, grad.ctypes.data))
        return ll.value, (logq[:self.n_strings] if want_logq else None), grad[:self.n]

    def upload_x(self, x):
        x = np.ascontiguousarray(x, dtype=np.float64)
        self._ck(self.L.wfsa_dev_upload_x(self.h, _p(x, F64P)))

    def eval_launch(self):
        self._ck(self.L.wfsa_dev_eval_launch(self.h))

    def sync(self):
        self._ck(self.L.wfsa_dev_sync(self.h))

    def eval_fetch(self, want_logq=False):
        ll = C.c_double()
        grad = np.zeros(max(self.n, 1))
        logq = np.zeros(max(self.n_strings, 1)) if want_logq else None
        self._ck(self.L.wfsa_dev_eval_fetch(self.h, C.byref(ll), _p(logq, F64P), _p(grad, F64P)))
        if want_logq:
            return ll.value, logq[:self.n_strings], grad[:self.n]
        return ll.value, grad[:self.n]

    def viterbi(self, x):
        """Most probable path of every string at x: (logw, path_off, trans_edge, emis_edge); the steps of string s are
        [path_off[s], path_off[s+1]) (descriptor edge ids; emis_edge -1 on the final transition), logw[s] = -inf: none."""
        return _viterbi(self.L, self.h, x, self.n_strings)

    def nbest(self, x, k):
        """The k most probable paths of every string at x: (logw [n_strings, k], path_off, trans_edge, emis_edge); path
        i = s * k + r is the r-th most probable path of string s, its steps [path_off[i], path_off[i+1]) as in viterbi,
        logw[s, r] = -inf: string s has at most r paths."""
        logw, off, tr, em = _viterbi(self.L, self.h, x, self.n_strings, k)
        return logw.reshape(self.n_strings, k), off, tr, em

    def sample(self, x, n, seed=0):
        """n independent draws from the path posterior of every string at x: (logw [n_strings, n], logq, path_off,
        trans_edge, emis_edge); path i = s * n + r is draw r of string s, its steps [path_off[i], path_off[i+1]) as in viterbi,
        logw[s, r] = -inf: string s has no path; logq[s] = log q_s from the sampler's forward sweep."""
        return _sample(self.L, self.h, x, self.n_strings, n, seed)

    def timer_begin(self):
        self._ck(self.L.wfsa_dev_timer_begin(self.h))

    def timer_begin_steps(self):
        self._ck(self.L.wfsa_dev_timer_begin_steps(self.h))

    def timer_end(self):
        ms = C.c_float()
        self._ck(self.L.wfsa_dev_timer_end(self.h, C.byref(ms)))
        return ms.value

    def timer_kernel_ms(self):
        ms, n = C.c_float(), C.c_int64()
        self._ck(self.L.wfsa_dev_timer_kernel_ms(self.h, C.byref(ms), C.byref(n)))
        return ms.value, n.value

    def timer_step_ms(self):
        """(sum of the per-evaluation device times since timer_begin, number of evaluations)"""
        ms, n = C.c_float(), C.c_int64()
        self._ck(self.L.wfsa_dev_timer_step_ms(self.h, C.byref(ms), C.byref(n)))
        return ms.value, n.value

    def timer_phase_ms(self):
        out = (C.c_float * 3)()
        self._ck(self.L.wfsa_dev_timer_phase_ms(self.h, out))
        return [out[0], out[1], out[2]]

    def eval6_phases(self, reset=True):
        """ns CTA 0 of k_eval6 spent in [weights, region types, grid barrier, fold + exchange] since the last reset"""
        out = np.zeros(4)
        self._ck(self.L.wfsa_dev_eval6_phases(self.h, _p(out, F64P), 1 if reset else 0))
        return out

    def rank_barrier(self):
        self._ck(self.L.wfsa_dev_rank_barrier(self.h))

    def l2_flush(self):
        self._ck(self.L.wfsa_dev_l2_flush(self.h))

    def timer_split_ms(self):
        a, b = C.c_float(), C.c_float()
        self._ck(self.L.wfsa_dev_timer_split_ms(self.h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def info(self):
        i = DevInfo()
        self._ck(self.L.wfsa_dev_get_info(self.h, C.byref(i)))
        return {k: getattr(i, k) for k, _ in DevInfo._fields_}

    def allreduce(self, values, op=0):
        v = np.ascontiguousarray(values, dtype=np.float64)
        self._ck(self.L.wfsa_dev_allreduce_f64(self.h, _p(v, F64P), len(v), op))
        return v

    def close(self):
        if self.h:
            self.L.wfsa_dev_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _sample(L, h, x, n_strings, n, seed):
    """wfsa_dev_sample, then the steps: (logw [n_strings, n], logq, path_off, trans_edge, emis_edge)."""
    def ck(rc):
        if rc != 0:
            raise WfsaError(rc, L.wfsa_dev_last_error(h).decode())
    x = np.ascontiguousarray(x, dtype=np.float64)
    logw = np.zeros(max(n_strings * n, 1))
    logq = np.zeros(max(n_strings, 1))
    off = np.zeros(n_strings * n + 1, dtype=np.int64)
    ck(L.wfsa_dev_sample(h, _p(x, F64P), n, seed, _p(logw, F64P), _p(logq, F64P), _p(off, I64P)))
    steps = max(int(off[-1]), 1)
    tr = np.zeros(steps, dtype=np.int32)
    em = np.zeros(steps, dtype=np.int32)
    ck(L.wfsa_dev_viterbi_paths(h, _p(tr, I32P), _p(em, I32P)))
    return logw[:n_strings * n].reshape(n_strings, n), logq[:n_strings], off, tr[:off[-1]], em[:off[-1]]


def philox4x32_10(ctr, key):
    """The Philox4x32-10 block function of wfsa_dev_sample (wfsa_philox4x32_10): 4 words out of a 4-word counter and a 2-word
    key."""
    c = np.ascontiguousarray(ctr, dtype=np.uint32); k = np.ascontiguousarray(key, dtype=np.uint32)
    out = np.zeros(4, dtype=np.uint32)
    lib().wfsa_philox4x32_10(_p(c, U32P), _p(k, U32P), _p(out, U32P))
    return out


def _viterbi(L, h, x, n_strings, k=None):
    """wfsa_dev_viterbi (k None) or wfsa_dev_nbest, then the steps: (logw, path_off, trans_edge, emis_edge) per path."""
    def ck(rc):
        if rc != 0:
            raise WfsaError(rc, L.wfsa_dev_last_error(h).decode())
    x = np.ascontiguousarray(x, dtype=np.float64)
    n_paths = n_strings * (k or 1)
    logw = np.zeros(max(n_paths, 1))
    off = np.zeros(n_paths + 1, dtype=np.int64)
    if k is None:
        ck(L.wfsa_dev_viterbi(h, _p(x, F64P), _p(logw, F64P), _p(off, I64P)))
    else:
        ck(L.wfsa_dev_nbest(h, _p(x, F64P), k, _p(logw, F64P), _p(off, I64P)))
    steps = max(int(off[-1]), 1)
    tr = np.zeros(steps, dtype=np.int32)
    em = np.zeros(steps, dtype=np.int32)
    ck(L.wfsa_dev_viterbi_paths(h, _p(tr, I32P), _p(em, I32P)))
    return logw[:n_paths], off, tr[:off[-1]], em[:off[-1]]


class Session:
    """The reference executable's flow (src/main.cpp:121-347) one call at a time, C++ host code underneath."""

    def __init__(self, fsa_text, corpus_text, optimizer="QuasiNewton", device=0, force_kernel=0, accum_mode=0,
                 accum_variant=0, rank=0, nranks=1, unique_id=None):
        self.L = lib()
        fa = fsa_text.encode("latin-1") if isinstance(fsa_text, str) else fsa_text
        co = corpus_text.encode("latin-1") if isinstance(corpus_text, str) else corpus_text
        self._uid = C.create_string_buffer(bytes(unique_id), UNIQUE_ID_BYTES) if unique_id is not None else None
        opt = SessionOptions(device, force_kernel, accum_mode, accum_variant, rank, nranks,
                             C.cast(self._uid, C.c_void_p) if self._uid is not None else None)
        self.h = C.c_void_p()
        rc = self.L.wfsa_session_create(fa, len(fa), co, len(co), optimizer.encode(), C.byref(opt), C.byref(self.h))
        if rc != 0:
            raise WfsaError(rc, self.L.wfsa_session_error(None).decode("latin-1"))
        self.optimizer = optimizer
        self.n = self.L.wfsa_session_n(self.h)
        self.k = self.L.wfsa_session_k(self.h)

    def _ck(self, rc):
        if rc != 0:
            raise WfsaError(rc, self.L.wfsa_session_error(self.h).decode("latin-1"))

    def describe(self):
        return json.loads(self.L.wfsa_session_describe(self.h).decode("latin-1"))

    def init(self, flags, x=None):
        xx = None if x is None else np.ascontiguousarray(x, dtype=np.float64)
        self._ck(self.L.wfsa_session_init(self.h, flags, _p(xx, F64P)))

    def eval(self, x=None, want_logq=True):
        xx = None if x is None else np.ascontiguousarray(x, dtype=np.float64)
        kl, ll = C.c_double(), C.c_double()
        grad = np.zeros(max(self.n, 1))
        nrec = self.L.wfsa_session_n_recognised_local(self.h)
        logq = np.zeros(max(nrec, 1)) if want_logq else None
        self._ck(self.L.wfsa_session_eval(self.h, _p(xx, F64P), C.byref(kl), C.byref(ll), _p(grad, F64P), _p(logq, F64P)))
        return {"kl": kl.value, "loglik": ll.value, "grad": grad[:self.n], "logq": None if logq is None else logq[:nrec]}

    def hessian(self, x=None):
        xx = None if x is None else np.ascontiguousarray(x, dtype=np.float64)
        H = np.zeros((max(self.n, 1), max(self.n, 1)))
        self._ck(self.L.wfsa_session_hessian(self.h, _p(xx, F64P), _p(H, F64P)))
        return H[:self.n, :self.n]

    def step(self, eta=1.0):
        info = np.zeros(9)
        n = C.c_int()
        self._ck(self.L.wfsa_session_step(self.h, eta, _p(info, F64P), C.byref(n)))
        return info[:n.value]

    def halt(self, tol):
        h = C.c_int()
        self._ck(self.L.wfsa_session_halt(self.h, tol, C.byref(h)))
        return bool(h.value)

    def x(self, with_multipliers=False):
        cnt = self.n + (self.k if with_multipliers else 0)
        v = np.zeros(max(cnt, 1))
        self._ck(self.L.wfsa_session_get_x(self.h, _p(v, F64P), cnt))
        return v[:cnt]

    def renormalize(self):
        self._ck(self.L.wfsa_session_renormalize(self.h))

    def result(self):
        v = np.zeros(8)
        self._ck(self.L.wfsa_session_result(self.h, _p(v, F64P)))
        return v

    def dump(self, full_precision=True):
        return self.L.wfsa_session_dump(self.h, 1 if full_precision else 0).decode("latin-1")

    def viterbi(self, x=None):
        """Device.viterbi on the session's backend, at x or the current weights, for every string of this shard."""
        return _viterbi(self.L, self.L.wfsa_session_backend(self.h), self.x() if x is None else x, self.backend_info()["n_strings"])

    def nbest(self, k, x=None):
        """Device.nbest on the session's backend, at x or the current weights, for every string of this shard."""
        ns = self.backend_info()["n_strings"]
        logw, off, tr, em = _viterbi(self.L, self.L.wfsa_session_backend(self.h), self.x() if x is None else x, ns, k)
        return logw.reshape(ns, k), off, tr, em

    def sample(self, n, seed=0, x=None):
        """Device.sample on the session's backend, at x or the current weights, for every string of this shard."""
        return _sample(self.L, self.L.wfsa_session_backend(self.h), self.x() if x is None else x,
                       self.backend_info()["n_strings"], n, seed)

    def backend_info(self):
        i = DevInfo()
        self.L.wfsa_dev_get_info(self.L.wfsa_session_backend(self.h), C.byref(i))
        return {k: getattr(i, k) for k, _ in DevInfo._fields_}

    def close(self):
        if self.h:
            self.L.wfsa_session_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
