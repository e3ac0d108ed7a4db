"""ctypes face of the CPU checker (oracle/liboracle.so) and, when present, of the compiled
reference sources (oracle/_ref/libnemo_ref.so). TEST INFRASTRUCTURE: import only from tests/,
__graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_DIR = os.path.dirname(os.path.abspath(__file__))
# Optional checkout of the reference project (nemotron-speech.cpp). Only the differential tests that compile or run the reference's
# own sources use it; they skip without it, and the committed fixtures under tests/golden/ stand in for it.
REFERENCE_DIR = os.environ.get("NSB_REFERENCE_DIR", "")
MM_REF, MM_F16, MM_BF16, MM_Q8FAST = 0, 1, 2, 3
KV_F32, KV_F16, KV_BF16 = 0, 1, 2

_f32p = np.ctypeslib.ndpointer(dtype=np.float32, flags="C_CONTIGUOUS")
_i16p = np.ctypeslib.ndpointer(dtype=np.int16, flags="C_CONTIGUOUS")
_i32p = np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS")


def reference_file(rel: str) -> str | None:
    """Path of `rel` inside the reference checkout, or None when there is no checkout or it lacks the file."""
    p = os.path.join(REFERENCE_DIR, rel) if REFERENCE_DIR else ""
    return p if p and os.path.exists(p) else None


def build(force: bool = False) -> None:
    so = os.path.join(_DIR, "liboracle.so")
    src = os.path.join(_DIR, "stream_oracle.cpp")
    stale = (not os.path.exists(so)) or os.path.getmtime(so) < os.path.getmtime(src)
    if force or stale or (reference_file("src") and not os.path.exists(os.path.join(_DIR, "_ref", "libnemo_ref.so"))):
        subprocess.check_call(["make", "-C", _DIR, "all"], stdout=subprocess.DEVNULL)


_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(os.path.join(_DIR, "liboracle.so"))
        L.orc_model_load.restype = C.c_void_p
        L.orc_model_load.argtypes = [C.c_char_p, C.c_int, C.c_int]
        L.orc_model_free.argtypes = [C.c_void_p]
        L.orc_model_n_layers.argtypes = [C.c_void_p]
        L.orc_model_vocab.restype = C.c_void_p
        L.orc_model_vocab.argtypes = [C.c_void_p]
        L.orc_pp_new.restype = C.c_void_p
        L.orc_pp_new.argtypes = [C.c_void_p]
        L.orc_pp_new_from_data.restype = C.c_void_p
        L.orc_pp_new_from_data.argtypes = [_f32p, _f32p]
        L.orc_pp_free.argtypes = [C.c_void_p]
        L.orc_pp_process.argtypes = [C.c_void_p, _i16p, C.c_int, _f32p, C.c_int]
        L.orc_subsampling.argtypes = [C.c_void_p, _f32p, C.c_int, _f32p, C.c_int]
        L.orc_matmul.argtypes = [C.c_void_p, C.c_char_p, _f32p, C.c_int, _f32p]
        L.orc_layer_norm.argtypes = [_f32p, C.c_int, C.c_int, _f32p, _f32p, _f32p]
        L.orc_pos_emb_row.argtypes = [C.c_int, _f32p]
        L.orc_stream_new.restype = C.c_void_p
        L.orc_stream_new.argtypes = [C.c_void_p, C.c_int]
        L.orc_stream_free.argtypes = [C.c_void_p]
        L.orc_stream_set_trace.argtypes = [C.c_void_p, C.c_int]
        L.orc_stream_push.argtypes = [C.c_void_p, _i16p, C.c_int]
        L.orc_stream_push_mel.argtypes = [C.c_void_p, _f32p, C.c_int]
        L.orc_stream_n_tokens.argtypes = [C.c_void_p]
        L.orc_stream_tokens.argtypes = [C.c_void_p, _i32p, C.c_int]
        L.orc_stream_chunks.argtypes = [C.c_void_p]
        L.orc_stream_cache_valid.argtypes = [C.c_void_p]
        L.orc_trace_enc.argtypes = [C.c_void_p, C.c_int, _f32p, C.c_int]
        L.orc_trace_n_evals.argtypes = [C.c_void_p]
        L.orc_trace_logits.argtypes = [C.c_void_p, C.c_int, _f32p, C.c_int]
        L.orc_trace_eval_token.argtypes = [C.c_void_p, C.c_int]
        L.orc_last_sub.argtypes = [C.c_void_p, _f32p, C.c_int]
        L.orc_last_mel.argtypes = [C.c_void_p, _f32p, C.c_int]
        L.orc_last_layer.argtypes = [C.c_void_p, C.c_int, _f32p, C.c_int]
        L.orc_get_cache.argtypes = [C.c_void_p, C.c_int, C.c_int, _f32p, C.c_int]
        L.orc_detok.argtypes = [C.c_void_p, _i32p, C.c_int, C.c_char_p, C.c_int]
        L.orc_transcribe_full.argtypes = [C.c_void_p, _f32p, C.c_int, _f32p, C.c_int, _i32p, _i32p, C.c_int, C.POINTER(C.c_int)]
        L.orc_set_threads.argtypes = [C.c_int]
        _lib = L
    return _lib


class Model:
    def __init__(self, gguf_path: str, mm_mode: int = MM_REF, kv_mode: int = KV_F32):
        self.h = lib().orc_model_load(gguf_path.encode(), mm_mode, kv_mode)
        if not self.h:
            raise RuntimeError(f"oracle: failed to load {gguf_path}")
        self.n_layers = lib().orc_model_n_layers(self.h)

    def close(self):
        if self.h:
            lib().orc_model_free(self.h)
            self.h = None

    def matmul(self, name: str, x: np.ndarray) -> np.ndarray:
        x = np.ascontiguousarray(x, dtype=np.float32)
        rows = x.shape[0]
        y = np.empty((rows, 8192), dtype=np.float32)
        n_out = lib().orc_matmul(self.h, name.encode(), x, rows, y.reshape(-1))
        assert n_out > 0, name
        return y.reshape(-1)[: rows * n_out].reshape(rows, n_out).copy()

    def subsampling(self, mel: np.ndarray) -> np.ndarray:
        mel = np.ascontiguousarray(mel, dtype=np.float32)
        out = np.empty((mel.shape[0], 1024), dtype=np.float32)
        rows = lib().orc_subsampling(self.h, mel, mel.shape[0], out, out.shape[0])
        assert rows > 0
        return out[:rows].copy()

    def transcribe_full(self, mel: np.ndarray):
        """Non-streaming batch path (nemo_encode, nemo-ggml.cpp:1467-1535) on a whole mel [M,128]:
        returns (encoder output [T,1024], token ids, encoder frame of each token)."""
        mel = np.ascontiguousarray(mel, dtype=np.float32)
        cap_rows = mel.shape[0] // 8 + 4
        enc = np.empty((cap_rows, 1024), dtype=np.float32)
        toks = np.empty(cap_rows * 10, dtype=np.int32); frames = np.empty_like(toks); n = C.c_int(0)
        T = lib().orc_transcribe_full(self.h, mel.reshape(-1), mel.shape[0], enc.reshape(-1), cap_rows, toks, frames, len(toks), C.byref(n))
        assert T >= 0, T
        return enc[:T].copy(), toks[:n.value].copy(), frames[:n.value].copy()

    def detok(self, toks) -> str:
        t = np.ascontiguousarray(toks, dtype=np.int32)
        buf = C.create_string_buffer(16 * max(1, len(t)) + 16)
        n = lib().orc_detok(self.h, t, len(t), buf, len(buf))
        assert n >= 0
        return buf.raw[:n].decode("utf-8")


class Preproc:
    def __init__(self, model: Model | None = None, fb: np.ndarray | None = None, window: np.ndarray | None = None):
        if model is not None:
            self.h = lib().orc_pp_new(model.h)
        else:
            self.h = lib().orc_pp_new_from_data(np.ascontiguousarray(fb, np.float32).reshape(-1),
                                                np.ascontiguousarray(window, np.float32))

    def process(self, pcm: np.ndarray) -> np.ndarray:
        pcm = np.ascontiguousarray(pcm, dtype=np.int16)
        cap = len(pcm) // 160 + 8
        out = np.empty((cap, 128), dtype=np.float32)
        n = lib().orc_pp_process(self.h, pcm, len(pcm), out.reshape(-1), cap)
        assert n >= 0
        return out[:n].copy()

    def __del__(self):
        if getattr(self, "h", None):
            lib().orc_pp_free(self.h)
            self.h = None


class Stream:
    def __init__(self, model: Model, right_context: int, trace: bool = False):
        self.model = model
        self.T = 1 + right_context
        self.h = lib().orc_stream_new(model.h, right_context)
        lib().orc_stream_set_trace(self.h, 1 if trace else 0)

    def push(self, pcm: np.ndarray) -> int:
        pcm = np.ascontiguousarray(pcm, dtype=np.int16)
        return lib().orc_stream_push(self.h, pcm, len(pcm))

    def push_mel(self, mel: np.ndarray) -> int:
        mel = np.ascontiguousarray(mel, dtype=np.float32)
        return lib().orc_stream_push_mel(self.h, mel.reshape(-1), mel.shape[0])

    @property
    def chunks(self) -> int:
        return lib().orc_stream_chunks(self.h)

    def tokens(self) -> np.ndarray:
        n = lib().orc_stream_n_tokens(self.h)
        out = np.empty(max(n, 1), dtype=np.int32)
        lib().orc_stream_tokens(self.h, out, len(out))
        return out[:n].copy()

    def trace_enc(self, chunk: int) -> np.ndarray:
        out = np.empty((self.T, 1024), dtype=np.float32)
        assert lib().orc_trace_enc(self.h, chunk, out.reshape(-1), out.size) == out.size
        return out

    def n_evals(self) -> int:
        return lib().orc_trace_n_evals(self.h)

    def trace_logits(self, ev: int) -> np.ndarray:
        out = np.empty(1025, dtype=np.float32)
        assert lib().orc_trace_logits(self.h, ev, out, 1025) == 1025
        return out

    def eval_token(self, ev: int) -> int:
        return lib().orc_trace_eval_token(self.h, ev)

    def last_sub(self) -> np.ndarray:
        out = np.empty((self.T, 1024), dtype=np.float32)
        assert lib().orc_last_sub(self.h, out.reshape(-1), out.size) == out.size
        return out

    def last_mel(self) -> np.ndarray:
        M = 9 + 8 * self.T
        out = np.empty((M, 128), dtype=np.float32)
        assert lib().orc_last_mel(self.h, out.reshape(-1), out.size) == out.size
        return out

    def last_layer(self, l: int) -> np.ndarray:
        out = np.empty((self.T, 1024), dtype=np.float32)
        assert lib().orc_last_layer(self.h, l, out.reshape(-1), out.size) == out.size
        return out

    def cache(self, which: int, layer: int) -> np.ndarray:
        rows = 70 if which < 2 else 8
        out = np.empty((rows, 1024), dtype=np.float32)
        assert lib().orc_get_cache(self.h, which, layer, out.reshape(-1), out.size) == out.size
        return out

    def __del__(self):
        if getattr(self, "h", None):
            lib().orc_stream_free(self.h)
            self.h = None


# ------------------------------------------------------------------------------------------
# compiled reference sources (optional)
# ------------------------------------------------------------------------------------------
_ref = None


def ref_available() -> bool:
    return os.path.exists(os.path.join(_DIR, "_ref", "libnemo_ref.so"))


def ref():
    global _ref
    if _ref is None:
        build()
        R = C.CDLL(os.path.join(_DIR, "_ref", "libnemo_ref.so"))
        R.ref_pp_new.restype = C.c_void_p
        R.ref_pp_new.argtypes = [_f32p, _f32p]
        R.ref_pp_free.argtypes = [C.c_void_p]
        R.ref_pp_process.argtypes = [C.c_void_p, _i16p, C.c_int, _f32p, C.c_int]
        R.ref_weights_load.restype = C.c_void_p
        R.ref_weights_load.argtypes = [C.c_char_p]
        R.ref_weights_free.argtypes = [C.c_void_p]
        R.ref_subsampling.argtypes = [C.c_void_p, _f32p, C.c_int, _f32p, C.c_int]
        R.ref_layer_forward.argtypes = [C.c_void_p, C.c_int, _f32p, C.c_int, _f32p]
        R.ref_cached_layer_step.argtypes = [C.c_void_p, C.c_int, _f32p, C.c_int, _f32p, C.c_int, _f32p, C.c_int, _f32p, _f32p, _f32p]
        R.ref_greedy.argtypes = [C.c_void_p, _f32p, C.c_int, _i32p, C.c_int]
        R.ref_joint_logits.argtypes = [C.c_void_p, _f32p, C.c_int, _f32p]
        _ref = R
    return _ref


class RefPreproc:
    def __init__(self, fb: np.ndarray, window: np.ndarray):
        self.h = ref().ref_pp_new(np.ascontiguousarray(fb, np.float32).reshape(-1), np.ascontiguousarray(window, np.float32))

    def process(self, pcm: np.ndarray) -> np.ndarray:
        pcm = np.ascontiguousarray(pcm, dtype=np.int16)
        cap = len(pcm) // 160 + 8
        out = np.empty((cap, 128), dtype=np.float32)
        n = ref().ref_pp_process(self.h, pcm, len(pcm), out.reshape(-1), cap)
        assert n >= 0
        return out[:n].copy()

    def __del__(self):
        if getattr(self, "h", None):
            ref().ref_pp_free(self.h)
            self.h = None


class RefWeights:
    def __init__(self, nemo_bin: str):
        self.h = ref().ref_weights_load(nemo_bin.encode())
        if not self.h:
            raise RuntimeError("reference weights load failed")

    def subsampling(self, mel: np.ndarray) -> np.ndarray:
        mel = np.ascontiguousarray(mel, dtype=np.float32)
        out = np.empty((mel.shape[0], 1024), dtype=np.float32)
        rows = ref().ref_subsampling(self.h, mel.reshape(-1), mel.shape[0], out.reshape(-1), out.shape[0])
        assert rows > 0
        return out[:rows].copy()

    def layer(self, l: int, x: np.ndarray) -> np.ndarray:
        x = np.ascontiguousarray(x, dtype=np.float32)
        y = np.empty_like(x)
        ref().ref_layer_forward(self.h, l, x.reshape(-1), x.shape[0], y.reshape(-1))
        return y

    def cached_layer_step(self, l: int, x: np.ndarray, att_hist: np.ndarray, conv_hist: np.ndarray):
        """One cached streaming step of layer l from the reference's compiled modules (ref_shim.cpp:ref_cached_layer_step).
        Returns (y, histories rolled forward: last 70 attention-input rows, last 8 conv-input rows)."""
        x = np.ascontiguousarray(x, dtype=np.float32)
        att_hist = np.ascontiguousarray(att_hist, dtype=np.float32).reshape(-1, 1024)
        conv_hist = np.ascontiguousarray(conv_hist, dtype=np.float32).reshape(-1, 1024)
        y, an, cn = np.empty_like(x), np.empty_like(x), np.empty_like(x)
        dummy = np.zeros(1, np.float32)
        ref().ref_cached_layer_step(self.h, l, x.reshape(-1), x.shape[0], att_hist.reshape(-1) if len(att_hist) else dummy, len(att_hist),
                                    conv_hist.reshape(-1) if len(conv_hist) else dummy, len(conv_hist), y.reshape(-1), an.reshape(-1), cn.reshape(-1))
        return y, np.concatenate([att_hist, an])[-70:], np.concatenate([conv_hist, cn])[-8:]

    def greedy(self, enc: np.ndarray) -> np.ndarray:
        enc = np.ascontiguousarray(enc, dtype=np.float32)
        out = np.empty(enc.shape[0] * 10 + 1, dtype=np.int32)
        n = ref().ref_greedy(self.h, enc.reshape(-1), enc.shape[0], out, len(out))
        return out[:n].copy()

    def joint_logits(self, enc_frame: np.ndarray, token: int) -> np.ndarray:
        out = np.empty(1025, dtype=np.float32)
        ref().ref_joint_logits(self.h, np.ascontiguousarray(enc_frame, np.float32), token, out)
        return out

    def __del__(self):
        if getattr(self, "h", None):
            ref().ref_weights_free(self.h)
            self.h = None
