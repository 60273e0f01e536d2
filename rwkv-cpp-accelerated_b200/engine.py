"""ctypes binding of the C ABI in include/rwkv_b200.h (tests + bench.py only).

Fails loudly: if the CUDA library has not been built, or no CUDA device is visible,
constructing an Engine raises EngineError. There is no CPU fallback.
"""
import ctypes
import os

import numpy as np

VOCAB = 50277
MODE_PARRALEL, MODE_GPT = 0, 1
GEN_GREEDY, GEN_TYPICAL = 0, 1

_PKG = os.path.dirname(os.path.abspath(__file__))
_LIB = None


class EngineError(RuntimeError):
    pass


def lib_path():
    # RWKV_B200_LIB: A/B-test another build of the same ABI (tools/sweep.py); default is the in-tree library
    return os.environ.get("RWKV_B200_LIB") or os.path.join(_PKG, "librwkv_b200.so")


def load_library():
    """dlopen librwkv_b200.so and declare every symbol of include/rwkv_b200.h."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = lib_path()
    if not os.path.exists(path):
        raise EngineError("CUDA extension not built: %s (run python __graft_entry__.py build)" % path)
    lib = ctypes.CDLL(path)
    c = ctypes
    ull, vp, cp, i32 = c.c_ulonglong, c.c_void_p, c.c_char_p, c.c_int
    pull, pdbl, pflt = c.POINTER(ull), c.POINTER(c.c_double), c.POINTER(c.c_float)
    sig = {
        "rwkv_b200_last_error": (cp, []),
        "rwkv_b200_abi_version": (i32, []),
        "rwkv_b200_device_count": (i32, []),
        "rwkv_b200_load": (i32, [cp, ull, i32, i32, c.POINTER(vp), pull, pull]),
        "rwkv_b200_load_tp": (i32, [cp, ull, i32, i32, i32, i32, c.POINTER(vp), pull, pull]),
        "rwkv_b200_free": (None, [vp]),
        "rwkv_b200_tensor": (vp, [vp, i32]),
        "rwkv_b200_n_layers": (ull, [vp]),
        "rwkv_b200_n_embed": (ull, [vp]),
        "rwkv_b200_max_gpt": (ull, [vp]),
        "rwkv_b200_host_alloc": (vp, [c.c_size_t]),
        "rwkv_b200_host_free": (None, [vp]),
        "rwkv_b200_state_upload": (i32, [vp, pdbl, pdbl, pdbl, pdbl, pdbl, ull]),
        "rwkv_b200_state_download": (i32, [vp, pdbl, pdbl, pdbl, pdbl, pdbl, ull]),
        "rwkv_b200_state_zero": (i32, [vp]),
        "rwkv_b200_forward": (i32, [vp, pull, ull, i32, pflt]),
        "rwkv_b200_forward_greedy": (i32, [vp, ull, pull, pflt]),
        "rwkv_b200_logits_host": (pflt, [vp]),
        "rwkv_b200_sample_typical": (i32, [vp, c.c_float, c.c_double, pull, pdbl]),
        "rwkv_b200_generate": (i32, [vp, ull, ull, i32, c.c_float, pdbl, pull, i32, pull, pull, pflt]),
        "rwkv_b200_debug_read": (c.c_longlong, [vp, cp, vp, c.c_size_t]),
        "rwkv_b200_decode_timed": (i32, [vp, pull, ull, i32, pflt]),
        "rwkv_b200_kernel_count": (i32, []),
        "rwkv_b200_kernel_name": (cp, [i32]),
        "rwkv_b200_profile": (i32, [vp, pull, ull, pflt, pull, pdbl]),
        "rwkv_b200_launch_count": (ull, [vp]),
        "rwkv_b200_set_option": (i32, [vp, cp, cp]),
        "rwkv_b200_tp_buffer_bytes": (c.c_size_t, [vp]),
        "rwkv_b200_tp_export": (i32, [vp, vp]),
        "rwkv_b200_tp_import": (i32, [vp, vp]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)  # AttributeError if a declared symbol is missing
        fn.restype = res
        fn.argtypes = args
    lib._declared = sorted(sig)
    _LIB = lib
    return lib


def _ptr(a, ctype):
    return a.ctypes.data_as(ctypes.POINTER(ctype)) if a is not None else None


class Engine:
    """One loaded model on one GPU. Mirrors the reference's RWKV host class at the
    granularity the tests need: load, forward(tokens, mode), host<->device state."""

    def __init__(self, path, max_gpt=1, device=0, quiet=True, tp_rank=0, tp_size=1):
        """tp_size > 1: this process is rank `tp_rank` of a tensor-parallel group (one GPU per rank); wire the
        ranks with tp.connect(engine) before the first forward (include/rwkv_b200.h, "tensor-parallel wiring")."""
        self.lib = load_library()
        if self.lib.rwkv_b200_device_count() <= 0:
            raise EngineError("no CUDA device visible; the B200 engine has no CPU fallback")
        h = ctypes.c_void_p()
        L, E = ctypes.c_ulonglong(), ctypes.c_ulonglong()
        rc = self.lib.rwkv_b200_load_tp(path.encode(), max_gpt, device, 1 if quiet else 0, tp_rank, tp_size,
                                        ctypes.byref(h), ctypes.byref(L), ctypes.byref(E))
        if rc != 0:
            raise EngineError("rwkv_b200_load(%s) failed [%d]: %s" % (path, rc, self._err()))
        self.h = h
        self.n_layers, self.n_embed, self.max_gpt = L.value, E.value, max_gpt
        self.tp_rank, self.tp_size = tp_rank, tp_size

    # -- tensor-parallel wiring ------------------------------------------------------------
    def tp_export(self):
        """CUDA IPC handle (64 bytes) of this rank's exchange block."""
        buf = (ctypes.c_ubyte * 64)()
        self._ck(self.lib.rwkv_b200_tp_export(self.h, ctypes.cast(buf, ctypes.c_void_p)), "tp_export")
        return bytes(buf)

    def tp_import(self, handles):
        """handles: one 64-byte handle per rank, in rank order (the own entry is ignored)."""
        if len(handles) != self.tp_size or any(len(x) != 64 for x in handles):
            raise EngineError("tp_import needs %d handles of 64 bytes" % self.tp_size)
        blob = b"".join(handles)
        buf = (ctypes.c_ubyte * len(blob)).from_buffer_copy(blob)
        self._ck(self.lib.rwkv_b200_tp_import(self.h, ctypes.cast(buf, ctypes.c_void_p)), "tp_import")

    def _err(self):
        return self.lib.rwkv_b200_last_error().decode(errors="replace")

    def _ck(self, rc, what):
        if rc != 0:
            raise EngineError("%s failed [%d]: %s" % (what, rc, self._err()))

    def close(self):
        if getattr(self, "h", None):
            self.lib.rwkv_b200_free(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- compute ---------------------------------------------------------------------------
    def forward(self, tokens, mode=MODE_GPT, want_logits=True):
        toks = np.ascontiguousarray(np.atleast_1d(np.asarray(tokens, dtype=np.uint64)))
        out = np.empty((len(toks), VOCAB), np.float32) if want_logits else None
        self._ck(self.lib.rwkv_b200_forward(self.h, _ptr(toks, ctypes.c_ulonglong), len(toks), mode,
                                            _ptr(out, ctypes.c_float)), "forward")
        return out

    def sample_typical(self, temp, u):
        """Device sampler on the logits of the last forward: (token, margin) for the uniform `u`."""
        tok, margin = ctypes.c_ulonglong(), ctypes.c_double()
        self._ck(self.lib.rwkv_b200_sample_typical(self.h, temp, u, ctypes.byref(tok), ctypes.byref(margin)), "sample_typical")
        return int(tok.value), float(margin.value)

    def generate(self, first, n, how=GEN_TYPICAL, temp=0.9, uniforms=None, stop=(), want_logits=True):
        """rwkv_b200_generate: n steps of forward + pick (GEN_GREEDY: arg-max; GEN_TYPICAL: the typical sampler with
        uniforms[i] at step i) from token `first` on the device. Returns (tokens t1..tk, the last step's logits or None);
        k < n only when tk is in `stop`."""
        out = np.empty(max(int(n), 1), np.uint64)
        k = ctypes.c_ulonglong()
        u = None if uniforms is None else np.ascontiguousarray(uniforms, dtype=np.float64)
        if u is not None and u.size < n:
            raise EngineError("generate: %d uniforms for %d steps" % (u.size, n))
        st = np.ascontiguousarray(np.asarray(list(stop), dtype=np.uint64)) if len(stop) else None
        lg = np.empty(VOCAB, np.float32) if want_logits else None
        self._ck(self.lib.rwkv_b200_generate(self.h, int(first), int(n), int(how), float(temp), _ptr(u, ctypes.c_double),
                                             _ptr(st, ctypes.c_ulonglong), 0 if st is None else len(st),
                                             _ptr(out, ctypes.c_ulonglong), ctypes.byref(k), _ptr(lg, ctypes.c_float)),
                 "generate")
        return [int(t) for t in out[:k.value]], lg

    def forward_greedy(self, token, want_logits=False):
        nxt = ctypes.c_ulonglong()
        out = np.empty(VOCAB, np.float32) if want_logits else None
        self._ck(self.lib.rwkv_b200_forward_greedy(self.h, int(token), ctypes.byref(nxt),
                                                   _ptr(out, ctypes.c_float)), "forward_greedy")
        return (nxt.value, out) if want_logits else nxt.value

    # -- state -----------------------------------------------------------------------------
    def state_zero(self):
        self._ck(self.lib.rwkv_b200_state_zero(self.h), "state_zero")

    def state_download(self, slots=1):
        n = self.n_layers * self.n_embed * slots
        arrs = [np.empty(n, np.float64) for _ in range(5)]
        self._ck(self.lib.rwkv_b200_state_download(self.h, *[_ptr(a, ctypes.c_double) for a in arrs], slots),
                 "state_download")
        return dict(zip(("xy", "aa", "bb", "pp", "dd"), arrs))

    def state_upload(self, st, slots=1):
        arrs = [np.ascontiguousarray(st[k], np.float64) if st.get(k) is not None else None
                for k in ("xy", "aa", "bb", "pp", "dd")]
        self._ck(self.lib.rwkv_b200_state_upload(self.h, *[_ptr(a, ctypes.c_double) for a in arrs], slots),
                 "state_upload")

    # -- knobs / measurement ---------------------------------------------------------------
    def set_option(self, key, value):
        self._ck(self.lib.rwkv_b200_set_option(self.h, key.encode(), str(value).encode()), "set_option(%s)" % key)

    def debug_read(self, name):
        E = self.n_embed
        dt, n = {"x": (np.float64, E), "logits": (np.float32, VOCAB)}[name]
        a = np.empty(n, dt)
        got = self.lib.rwkv_b200_debug_read(self.h, name.encode(), a.ctypes.data_as(ctypes.c_void_p), a.nbytes)
        if got != n:
            raise EngineError("debug_read(%s) failed" % name)
        return a

    def read_trace(self, grid=148, per_cta=2048):
        """Per-CTA globaltimer stamps of the last token kernel (set_option('trace', 1) first)."""
        a = np.zeros(grid * per_cta, np.uint64)
        got = self.lib.rwkv_b200_debug_read(self.h, b"trace", a.ctypes.data_as(ctypes.c_void_p), a.nbytes)
        if got != a.size:
            raise EngineError("read_trace failed (trace option not enabled?)")
        return a.reshape(grid, per_cta)

    def read_tile_trace(self, grid=148, per_cta=4096):
        """[2][grid][per_cta] globaltimer: tile copy issued by the producer / tile seen ready by consumer thread 0."""
        a = np.zeros(2 * grid * per_cta, np.uint64)
        got = self.lib.rwkv_b200_debug_read(self.h, b"ptrace", a.ctypes.data_as(ctypes.c_void_p), a.nbytes)
        if got != a.size:
            raise EngineError("read_tile_trace failed")
        return a.reshape(2, grid, per_cta)

    def decode_timed(self, tokens, teacher_forced=True):
        toks = np.ascontiguousarray(np.asarray(tokens, dtype=np.uint64))
        ms = ctypes.c_float()
        self._ck(self.lib.rwkv_b200_decode_timed(self.h, _ptr(toks, ctypes.c_ulonglong), len(toks),
                                                 1 if teacher_forced else 0, ctypes.byref(ms)), "decode_timed")
        return ms.value

    def profile(self, tokens):
        k = self.lib.rwkv_b200_kernel_count()
        toks = np.ascontiguousarray(np.asarray(tokens, dtype=np.uint64))
        ms = np.zeros(k, np.float32)
        cnt = np.zeros(k, np.uint64)
        by = np.zeros(k, np.float64)
        self._ck(self.lib.rwkv_b200_profile(self.h, _ptr(toks, ctypes.c_ulonglong), len(toks),
                                            _ptr(ms, ctypes.c_float), _ptr(cnt, ctypes.c_ulonglong),
                                            _ptr(by, ctypes.c_double)), "profile")
        names = [self.lib.rwkv_b200_kernel_name(i).decode() for i in range(k)]
        return {n: {"ms_sum": float(ms[i]), "launches": int(cnt[i]), "bytes_per_launch": float(by[i])}
                for i, n in enumerate(names)}

    @property
    def launch_count(self):
        return int(self.lib.rwkv_b200_launch_count(self.h))
