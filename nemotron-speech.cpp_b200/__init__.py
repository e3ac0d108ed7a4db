"""Python face of libnsb200.so -- the B200-native streaming ASR engine (C ABI: include/nsb200.h).

ctypes only: the library is plain C ABI + CUDA runtime; torch is not involved in the data path.
Importing this module never falls back to anything: if the shared library is missing it raises,
and every compute call raises NsbError when no sm_100 GPU is usable.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_DIR, "libnsb200.so")

EPI_NONE, EPI_RELU, EPI_SILU, EPI_RESID, EPI_PARTIAL = 0, 1, 2, 3, 4
OUT_F32, OUT_F16, OUT_BF16 = 0, 1, 2
COMPUTE_AUTO, COMPUTE_F32, COMPUTE_F16, COMPUTE_BF16, COMPUTE_Q8_0, COMPUTE_Q8_0_STRICT = 0, 1, 2, 3, 4, 5
KV_F32, KV_F16, KV_BF16 = 0, 1, 2


class NsbError(RuntimeError):
    pass


class EngineConfig(C.Structure):
    _fields_ = [("device", C.c_int32), ("compute", C.c_int32), ("kv_dtype", C.c_int32), ("att_right_context", C.c_int32),
                ("max_streams", C.c_int32), ("use_cuda_graph", C.c_int32), ("decode_overlap", C.c_int32), ("reserved", C.c_int32 * 5)]


class Stats(C.Structure):
    _fields_ = [("steps", C.c_int64), ("chunks", C.c_int64), ("kernel_launches", C.c_int64), ("device_ms", C.c_double),
                ("last_step_ms", C.c_double)]


class TraceRecord(C.Structure):
    _fields_ = [("t", C.c_uint64 * 6), ("tag", C.c_int32), ("grid", C.c_int32)]


TRACE_TAGS = {1: "logmel", 2: "stem", 3: "dwconv", 4: "melhist", 5: "gemm_f32", 6: "gemm_tc", 7: "gemm_q8", 8: "ln", 9: "ln2", 10: "attn",
              11: "convmod", 12: "advance", 13: "decode", 14: "other"}


class GemmOp(C.Structure):
    _fields_ = [("weight", C.c_char_p), ("rows", C.c_int32), ("epi", C.c_int32), ("alpha", C.c_float), ("out_type", C.c_int32),
                ("splits", C.c_int32), ("c0", C.c_int32), ("c_group", C.c_int32), ("c_drop", C.c_int32), ("force_bn", C.c_int32),
                ("force_stages", C.c_int32), ("rotate", C.c_int32), ("bias", C.c_void_p), ("c_init", C.c_void_p)]


class ModelInfo(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("n_mels", "d_model", "n_heads", "d_head", "d_ff", "n_layers", "kernel_size", "vocab_size",
                                         "decoder_dim", "joint_dim", "n_tensors", "weight_type")] + [("vocab", C.c_char * (1025 * 8))]


EXPORTS = ["nsb_gguf_probe", "nsb_gguf_read_tensor", "nsb_default_config", "nsb_engine_create", "nsb_engine_destroy", "nsb_last_error", "nsb_engine_n_layers",
           "nsb_engine_vocab_size", "nsb_engine_vocab", "nsb_engine_chunk_samples", "nsb_engine_shift_samples", "nsb_engine_compute", "nsb_engine_set_cuda_graph",
           "nsb_stream_open", "nsb_stream_close", "nsb_stream_reset", "nsb_stream_push_pcm", "nsb_push_pcm_batch", "nsb_pop_tokens_batch", "nsb_stream_ready", "nsb_engine_step", "nsb_engine_step_begin", "nsb_engine_step_end",
           "nsb_engine_drain", "nsb_stream_pop_tokens", "nsb_stream_chunks", "nsb_detokenize", "nsb_engine_get_stats",
           "nsb_bench_prepare", "nsb_bench_step", "nsb_bench_steps", "nsb_bench_profile", "nsb_profiler_range", "nsb_bench_gemm", "nsb_trace_enable", "nsb_trace_fetch", "nsb_debug_enable", "nsb_debug_get", "nsb_debug_get_cache", "nsb_op_logmel",
           "nsb_op_gemm", "nsb_op_gemm_ex", "nsb_op_layernorm", "nsb_transcribe_full", "nsb_stream_export", "nsb_stream_import"]


def build(force: bool = False) -> str:
    """Compile libnsb200.so for sm_100a in-tree (nvcc cross-compiles without a GPU)."""
    if force or not os.path.exists(LIB_PATH):
        subprocess.check_call(["make", "-C", _DIR, "-j8", "all"], stdout=subprocess.DEVNULL)
    return LIB_PATH


_lib = None
_f32p = np.ctypeslib.ndpointer(dtype=np.float32, flags="C_CONTIGUOUS")
_i16p = np.ctypeslib.ndpointer(dtype=np.int16, flags="C_CONTIGUOUS")
_i32p = np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS")


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise NsbError(f"{LIB_PATH} is missing: run __graft_entry__.build() (there is no fallback path)")
        L = C.CDLL(LIB_PATH)
        vp, ci = C.c_void_p, C.c_int
        L.nsb_last_error.restype = C.c_char_p
        L.nsb_gguf_probe.argtypes = [C.c_char_p, C.POINTER(ModelInfo)]
        L.nsb_gguf_read_tensor.argtypes = [C.c_char_p, C.c_char_p, C.c_void_p, C.c_size_t, C.POINTER(C.c_int)]
        L.nsb_gguf_read_tensor.restype = C.c_longlong
        L.nsb_default_config.argtypes = [C.POINTER(EngineConfig)]
        L.nsb_engine_create.argtypes = [C.c_char_p, C.POINTER(EngineConfig), C.POINTER(vp)]
        L.nsb_engine_destroy.argtypes = [vp]
        for n in ("nsb_engine_n_layers", "nsb_engine_vocab_size", "nsb_engine_chunk_samples", "nsb_engine_shift_samples",
                  "nsb_engine_compute", "nsb_stream_open", "nsb_engine_step", "nsb_engine_step_begin", "nsb_engine_step_end", "nsb_engine_drain"):
            getattr(L, n).argtypes = [vp]
        L.nsb_engine_vocab.argtypes = [vp]
        L.nsb_engine_set_cuda_graph.argtypes = [vp, ci]
        L.nsb_engine_vocab.restype = vp
        for n in ("nsb_stream_close", "nsb_stream_reset", "nsb_stream_ready", "nsb_stream_chunks"):
            getattr(L, n).argtypes = [vp, ci]
        L.nsb_stream_export.argtypes = [vp, ci, vp, C.c_size_t]
        L.nsb_stream_export.restype = C.c_longlong
        L.nsb_stream_import.argtypes = [vp, C.c_char_p, C.c_size_t]
        L.nsb_stream_push_pcm.argtypes = [vp, ci, _i16p, ci]
        L.nsb_stream_pop_tokens.argtypes = [vp, ci, _i32p, ci]
        L.nsb_push_pcm_batch.argtypes = [vp, ci, _i32p, _i16p, ci, ci]
        L.nsb_pop_tokens_batch.argtypes = [vp, ci, _i32p, _i32p, ci, _i32p]
        L.nsb_detokenize.argtypes = [vp, _i32p, ci, C.c_char_p, ci]
        L.nsb_engine_get_stats.argtypes = [vp, C.POINTER(Stats)]
        L.nsb_bench_prepare.argtypes = [vp, ci, _i16p, ci, ci]
        L.nsb_bench_step.argtypes = [vp, C.POINTER(C.c_float)]
        L.nsb_bench_steps.argtypes = [vp, ci, C.POINTER(C.c_float), C.POINTER(C.c_float)]
        L.nsb_bench_profile.argtypes = [vp, C.POINTER(C.c_float), C.POINTER(C.c_int), C.POINTER(C.c_float)]
        L.nsb_profiler_range.argtypes = [ci]
        L.nsb_trace_enable.argtypes = [vp, ci]
        L.nsb_trace_fetch.argtypes = [vp, C.POINTER(TraceRecord), ci]
        L.nsb_bench_gemm.argtypes = [vp, ci, ci, ci, ci, ci, ci, ci, C.POINTER(C.c_float)]
        L.nsb_debug_enable.argtypes = [vp, ci]
        L.nsb_debug_get.argtypes = [vp, C.c_char_p, _f32p, C.c_size_t]
        L.nsb_debug_get_cache.argtypes = [vp, ci, ci, ci, _f32p, C.c_size_t]
        L.nsb_op_logmel.argtypes = [vp, _i16p, ci, ci, _f32p, C.c_size_t]
        L.nsb_op_gemm.argtypes = [vp, C.c_char_p, _f32p, ci, _f32p, C.c_size_t]
        L.nsb_op_gemm_ex.argtypes = [vp, C.POINTER(GemmOp), _f32p, vp, C.c_size_t, C.POINTER(C.c_longlong)]
        L.nsb_op_layernorm.argtypes = [vp, _f32p, ci, vp, ci, C.c_float, _f32p, _f32p, vp, vp, ci, ci, _f32p, vp]
        L.nsb_transcribe_full.argtypes = [vp, _i16p, ci, _i32p, _i32p, ci, C.POINTER(C.c_int), C.c_void_p, C.c_size_t]
        _lib = L
    return _lib


def _check(rc: int) -> int:
    if rc < 0:
        raise NsbError(f"nsb error {rc}: {lib().nsb_last_error().decode(errors='replace')}")
    return rc


def probe(path: str) -> ModelInfo:
    info = ModelInfo()
    _check(lib().nsb_gguf_probe(path.encode(), C.byref(info)))
    return info


def read_tensor(path: str, name: str):
    """(floats, ggml type) of one tensor as the engine's loader sees it (no GPU needed)."""
    t = C.c_int(0)
    n = _check(int(lib().nsb_gguf_read_tensor(path.encode(), name.encode(), None, 0, C.byref(t))))
    out = np.empty(n, dtype=np.float32)
    _check(int(lib().nsb_gguf_read_tensor(path.encode(), name.encode(), out.ctypes.data_as(C.c_void_p), out.size, C.byref(t))))
    return out, t.value


class Engine:
    """One engine per GPU: weights + per-stream caches resident in HBM; streams are slots."""

    def __init__(self, gguf_path: str, right_context: int = 0, max_streams: int = 1, compute: int = COMPUTE_AUTO,
                 kv_dtype: int = KV_F32, device: int = 0, cuda_graph: bool = True, decode_overlap: int = 0):
        cfg = EngineConfig()
        lib().nsb_default_config(C.byref(cfg))
        cfg.device, cfg.compute, cfg.kv_dtype = device, compute, kv_dtype
        cfg.att_right_context, cfg.max_streams = right_context, max_streams
        cfg.use_cuda_graph = 1 if cuda_graph else 0
        cfg.decode_overlap = decode_overlap                    # 0 auto (<= 128 token rows), 1 always, 2 never
        h = C.c_void_p()
        _check(lib().nsb_engine_create(gguf_path.encode(), C.byref(cfg), C.byref(h)))
        self.h = h
        self.T = 1 + right_context
        self.max_streams = max_streams
        self.n_layers = lib().nsb_engine_n_layers(h)
        self.chunk_samples = lib().nsb_engine_chunk_samples(h)
        self.shift_samples = lib().nsb_engine_shift_samples(h)
        self.compute = lib().nsb_engine_compute(h)

    def close(self):
        if getattr(self, "h", None):
            lib().nsb_engine_destroy(self.h)
            self.h = None

    __del__ = close

    def set_cuda_graph(self, on: bool):
        _check(lib().nsb_engine_set_cuda_graph(self.h, 1 if on else 0))

    # ---- streams ----
    def open_stream(self) -> int:
        return _check(lib().nsb_stream_open(self.h))

    def close_stream(self, s: int):
        _check(lib().nsb_stream_close(self.h, s))

    def reset_stream(self, s: int):
        _check(lib().nsb_stream_reset(self.h, s))

    def export_stream(self, s: int) -> bytes:
        """Snapshot of an open stream (nsb_stream_export, include/nsb200.h); the stream stays open and continues unchanged."""
        n = _check(int(lib().nsb_stream_export(self.h, s, None, 0)))
        buf = C.create_string_buffer(n)
        _check(int(lib().nsb_stream_export(self.h, s, buf, n)))
        return buf.raw

    def import_stream(self, blob: bytes) -> int:
        """A snapshot from export_stream as a new stream of this engine (nsb_stream_import); returns its id."""
        blob = bytes(blob)
        return _check(lib().nsb_stream_import(self.h, blob, len(blob)))

    def push(self, s: int, pcm: np.ndarray):
        pcm = np.ascontiguousarray(pcm, dtype=np.int16)
        if len(pcm):
            _check(lib().nsb_stream_push_pcm(self.h, s, pcm, len(pcm)))

    def push_batch(self, streams, pcm: np.ndarray):
        """pcm [n_streams, n_samples] int16: row i -> streams[i] (one C call)."""
        ids = np.ascontiguousarray(streams, dtype=np.int32)
        pcm = np.ascontiguousarray(pcm, dtype=np.int16)
        assert pcm.ndim == 2 and pcm.shape[0] == len(ids)
        if pcm.shape[1]:
            _check(lib().nsb_push_pcm_batch(self.h, len(ids), ids, pcm.reshape(-1), pcm.shape[1], pcm.shape[1]))

    def pop_tokens_batch(self, streams, cap_per_stream: int = 256):
        """-> (tokens [n_streams, cap], counts [n_streams]); call again while a count == cap."""
        ids = np.ascontiguousarray(streams, dtype=np.int32)
        out = np.empty((len(ids), cap_per_stream), dtype=np.int32)
        cnt = np.empty(len(ids), dtype=np.int32)
        _check(lib().nsb_pop_tokens_batch(self.h, len(ids), ids, out.reshape(-1), cap_per_stream, cnt))
        return out, cnt

    def ready(self, s: int) -> bool:
        return _check(lib().nsb_stream_ready(self.h, s)) == 1

    def step(self) -> int:
        return _check(lib().nsb_engine_step(self.h))

    def step_begin(self) -> int:
        return _check(lib().nsb_engine_step_begin(self.h))

    def step_end(self) -> int:
        return _check(lib().nsb_engine_step_end(self.h))

    def drain(self) -> int:
        return _check(lib().nsb_engine_drain(self.h))

    def pop_tokens(self, s: int) -> np.ndarray:
        out, buf = [], np.empty(1024, dtype=np.int32)
        while True:
            n = _check(lib().nsb_stream_pop_tokens(self.h, s, buf, len(buf)))
            if n == 0:
                break
            out.append(buf[:n].copy())
        return np.concatenate(out) if out else np.empty(0, dtype=np.int32)

    def chunks(self, s: int) -> int:
        return _check(lib().nsb_stream_chunks(self.h, s))

    def detok(self, toks) -> str:
        t = np.ascontiguousarray(toks, dtype=np.int32)
        buf = C.create_string_buffer(16 * max(1, len(t)) + 16)
        n = _check(lib().nsb_detokenize(self.h, t, len(t), buf, len(buf)))
        return buf.raw[:n].decode("utf-8")

    def stats(self) -> Stats:
        s = Stats()
        lib().nsb_engine_get_stats(self.h, C.byref(s))
        return s

    # ---- bench ----
    def bench_prepare(self, pcm: np.ndarray, warm_chunks: int):
        pcm = np.ascontiguousarray(pcm, dtype=np.int16)
        assert pcm.ndim == 2
        _check(lib().nsb_bench_prepare(self.h, pcm.shape[0], pcm.reshape(-1), pcm.shape[1], warm_chunks))

    def bench_step(self) -> float:
        ms = C.c_float()
        _check(lib().nsb_bench_step(self.h, C.byref(ms)))
        return ms.value

    def bench_steps(self, n: int):
        """n steps enqueued back to back; returns (total device ms, per-step device ms)."""
        per = (C.c_float * n)(); tot = C.c_float()
        _check(lib().nsb_bench_steps(self.h, n, per, C.byref(tot)))
        return tot.value, [float(x) for x in per]

    PROFILE_CLASSES = ("logmel", "subsampling", "layernorm", "layer_gemm", "attention", "conv_module", "decode", "misc")

    def bench_profile(self):
        """One bench step with per-launch CUDA events -> ({class: (ms, launches)}, total_ms)."""
        ms = (C.c_float * 8)()
        n = (C.c_int * 8)()
        tot = C.c_float()
        _check(lib().nsb_bench_profile(self.h, ms, n, C.byref(tot)))
        return {k: (ms[i], n[i]) for i, k in enumerate(self.PROFILE_CLASSES)}, tot.value

    def bench_gemm(self, kind: int, rows: int, bn: int, stages: int, splits: int = 1, rotate: int = 1, iters: int = 5) -> float:
        us = C.c_float()
        _check(lib().nsb_bench_gemm(self.h, kind, rows, bn, stages, splits, rotate, iters, C.byref(us)))
        return us.value

    def trace_enable(self, capacity: int):
        _check(lib().nsb_trace_enable(self.h, capacity))

    def trace_fetch(self, cap: int = 4096):
        buf = (TraceRecord * cap)()
        n = _check(lib().nsb_trace_fetch(self.h, buf, cap))
        return [(TRACE_TAGS.get(buf[i].tag, str(buf[i].tag)), buf[i].grid, [int(x) for x in buf[i].t]) for i in range(n)]

    # ---- debug / operators ----
    def debug_enable(self, on: bool = True):
        _check(lib().nsb_debug_enable(self.h, 1 if on else 0))

    def debug_get(self, name: str, B: int) -> np.ndarray:
        rows = self.max_streams * self.T
        if name == "mel":
            M = 9 + 8 * self.T
            buf = np.empty(self.max_streams * M * 128, dtype=np.float32)
            _check(lib().nsb_debug_get(self.h, name.encode(), buf, buf.size))
            return buf.reshape(self.max_streams, M, 128)[:B].copy()
        if name == "logits":
            buf = np.empty((11 * self.T) * 1025, dtype=np.float32)
            n = _check(lib().nsb_debug_get(self.h, name.encode(), buf, buf.size))
            return buf[:n].reshape(-1, 1025).copy()
        buf = np.empty(rows * 1024, dtype=np.float32)
        _check(lib().nsb_debug_get(self.h, name.encode(), buf, buf.size))
        return buf.reshape(rows, 1024)[: B * self.T].copy()

    def debug_cache(self, stream: int, which: int, layer: int) -> np.ndarray:
        rows = 70 if which < 2 else 8
        buf = np.empty(rows * 1024, dtype=np.float32)
        _check(lib().nsb_debug_get_cache(self.h, stream, which, layer, buf, buf.size))
        return buf.reshape(rows, 1024)

    def op_logmel(self, pcm: np.ndarray) -> np.ndarray:
        pcm = np.ascontiguousarray(pcm, dtype=np.int16)
        if pcm.ndim == 1:
            pcm = pcm[None]
        ns, n = pcm.shape
        nf = (256 + n - 512 + 160) // 160 if 256 + n >= 512 else 0
        out = np.empty((ns, max(nf, 1), 128), dtype=np.float32)
        got = _check(lib().nsb_op_logmel(self.h, pcm.reshape(-1), ns, n, out.reshape(-1), out.size))
        assert got == nf, (got, nf)
        return out[:, :nf]

    def op_gemm(self, weight_name: str, x: np.ndarray) -> np.ndarray:
        x = np.ascontiguousarray(x, dtype=np.float32)
        y = np.empty((x.shape[0], 4096), dtype=np.float32)
        n_out = _check(lib().nsb_op_gemm(self.h, weight_name.encode(), x, x.shape[0], y.reshape(-1), y.size))
        return y.reshape(-1)[: x.shape[0] * n_out].reshape(x.shape[0], n_out).copy()

    def op_gemm_ex(self, weight_name: str, x: np.ndarray, *, epi: int = EPI_NONE, alpha: float = 1.0, bias=None, out_type: int = OUT_F32,
                   splits: int = 1, c0: bool = False, c_group: int = 0, c_drop: int = 0, force_bn: int = 0, force_stages: int = 0,
                   rotate: int = 1, c_init=None):
        """One GEMM of the step as an operator (nsb_op_gemm_ex, include/nsb200.h) -> (y, guard_bad). y: [m_out, n_out] float32, or
        uint16 bits for 16-bit outputs; EPI_PARTIAL: every k-slice plane [splits, m_out, n_out] float32 (plane 0 from C0 when c0)."""
        x = np.ascontiguousarray(x, dtype=np.float32)
        rows = x.shape[0]
        m_out = rows // c_group * (c_group - c_drop) if c_group else rows
        keep = []
        def ptr(a):
            if a is None:
                return None
            a = np.ascontiguousarray(a, dtype=np.float32); keep.append(a)
            return a.ctypes.data_as(C.c_void_p)
        op = GemmOp(weight_name.encode(), rows, epi, alpha, out_type, splits, int(c0), c_group, c_drop, force_bn, force_stages, rotate,
                    ptr(bias), ptr(c_init))
        n_cap = 4096
        shape = (splits, m_out, n_cap) if epi == EPI_PARTIAL else (m_out, n_cap)
        y = np.empty(shape, dtype=np.float32 if out_type == OUT_F32 else np.uint16)
        bad = C.c_longlong(-1)
        n = _check(lib().nsb_op_gemm_ex(self.h, C.byref(op), x, y.ctypes.data_as(C.c_void_p), y.nbytes, C.byref(bad)))
        y = y.reshape(-1)[: int(np.prod(shape[:-1])) * n].reshape(shape[:-1] + (n,)).copy()
        return y, bad.value

    def op_layernorm(self, x: np.ndarray, g1, b1, *, planes=None, alpha: float = 1.0, fused: bool = False, g2=None, b2=None,
                     out_type: int = OUT_F32):
        """The step's LayerNorm launch (nsb_op_layernorm, include/nsb200.h) -> (x after the launch, y float32 or uint16 bits)."""
        x = np.ascontiguousarray(x, dtype=np.float32)
        rows = x.shape[0]
        f = lambda a: None if a is None else np.ascontiguousarray(a, dtype=np.float32)
        planes, g1, b1, g2, b2 = f(planes), f(g1), f(b1), f(g2), f(b2)
        vp = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)
        x_out = np.empty_like(x)
        y = np.zeros((rows, 1024), dtype=np.float32 if out_type == OUT_F32 else np.uint16)
        n_planes = 0 if planes is None else planes.shape[0]
        _check(lib().nsb_op_layernorm(self.h, x, rows, vp(planes), n_planes, alpha, g1, b1, vp(g2), vp(b2), int(fused), out_type, x_out,
                                      y.ctypes.data_as(C.c_void_p)))
        return x_out, y

    def transcribe_full(self, pcm: np.ndarray, want_enc: bool = True, want_frames: bool = False):
        """Non-streaming batch path (nsb_transcribe_full, include/nsb200.h): one whole utterance ->
        (token ids, encoder output [frames, 1024] or None[, encoder frame of each token])."""
        pcm = np.ascontiguousarray(pcm, dtype=np.int16)
        frames_cap = len(pcm) // 1280 + 8
        toks = np.empty(10 * frames_cap, dtype=np.int32)
        frm = np.empty(10 * frames_cap, dtype=np.int32)
        enc = np.empty((frames_cap, 1024), dtype=np.float32) if want_enc else None
        nf = C.c_int(0)
        n = _check(lib().nsb_transcribe_full(self.h, pcm, len(pcm), toks, frm, len(toks), C.byref(nf),
                                             enc.ctypes.data_as(C.c_void_p) if want_enc else None, enc.size if want_enc else 0))
        out = (toks[:n].copy(), (enc[:nf.value].copy() if want_enc else None))
        return out + (frm[:n].copy(),) if want_frames else out
