#!/usr/bin/env python3
"""Synthetic assets for the streaming hot path: seeded model weights written as GGUF v3
(f32 / f16 / q8_0) and as the reference's "NEMO" v1 .bin, plus seeded 16 kHz s16le PCM.

There are no real weights and no network in this environment, so every parity / bench run
uses these. The *layout* written here is the contract, not the values:

  * GGUF: KV order, tensor names, reversed dims, 32-byte alignment and *which tensors get
    quantised* follow the reference converter (scripts/convert_to_gguf.py:296-308 hparams,
    :322-388 tensor prep incl. pointwise squeeze / depthwise squeeze+transpose, :221-238 +
    :346-352 quantise rule, :93-129 Q8_0 block = fp16 d + 32 x int8 with q = round(x / fp16(d)),
    :407-447 file writer).
  * NEMO bin: scripts/convert_weights.py:36-58,73-77 (magic "NEMO", version 1, per tensor
    name/ndims/dims/dtype/data, PyTorch shapes) -- consumed by src/reference/ggml_weights.cpp:19-157.

Everything is generated tensor-by-tensor from a per-tensor seed so that the f32 / f16 / q8_0 /
NEMO files of one (seed, n_layers) hold the same underlying values.
"""
from __future__ import annotations

import argparse
import os
import re
import struct
import tempfile
import zlib

import numpy as np

GGUF_MAGIC = b"GGUF"
GGUF_VERSION = 3
ALIGN = 32
T_U32, T_STR = 4, 8
GGML_F32, GGML_F16, GGML_Q4_0, GGML_Q8_0 = 0, 1, 2, 8

D_MODEL, D_FF, N_HEADS, D_HEAD = 1024, 4096, 8, 128
N_MELS, N_BINS, WIN = 128, 257, 400
VOCAB, HID, JOINT = 1025, 640, 640
KSIZE = 9
BRANCH_GAIN = float(os.environ.get("NSB_BRANCH_GAIN", 0.15))
ENC_GAIN = float(os.environ.get("NSB_ENC_GAIN", 4.0))
PRED_GAIN = float(os.environ.get("NSB_PRED_GAIN", 1.0))
SUB_CH, SUB_W = 256, 17

QUANT_RE = re.compile(r"encoder\.layers\.\d+\.(feed_forward\d+|self_attn|conv)\.[^.]+\.weight$")
DW_RE = re.compile(r"\.conv\.depthwise_conv\.weight$")
PW_RE = re.compile(r"\.conv\.(pointwise_conv1|pointwise_conv2)\.weight$")


# --------------------------------------------------------------------------------------
# tensor inventory (PyTorch shapes, as a .nemo checkpoint holds them)
# --------------------------------------------------------------------------------------
def tensor_specs(n_layers: int):
    """Yield (name, torch_shape, kind). kind drives the init distribution."""
    pe = "encoder.pre_encode."
    yield pe + "conv.0.weight", (SUB_CH, 1, 3, 3), ("w0", 9)
    yield pe + "conv.0.bias", (SUB_CH,), ("b", 0)
    yield pe + "conv.2.weight", (SUB_CH, 1, 3, 3), ("w", 9)
    yield pe + "conv.2.bias", (SUB_CH,), ("b", 0)
    yield pe + "conv.3.weight", (SUB_CH, SUB_CH, 1, 1), ("w", SUB_CH)
    yield pe + "conv.3.bias", (SUB_CH,), ("b", 0)
    yield pe + "conv.5.weight", (SUB_CH, 1, 3, 3), ("w", 9)
    yield pe + "conv.5.bias", (SUB_CH,), ("b", 0)
    yield pe + "conv.6.weight", (SUB_CH, SUB_CH, 1, 1), ("w", SUB_CH)
    yield pe + "conv.6.bias", (SUB_CH,), ("b", 0)
    yield pe + "out.weight", (D_MODEL, SUB_CH * SUB_W), ("w", SUB_CH * SUB_W)
    yield pe + "out.bias", (D_MODEL,), ("b", 0)
    for i in range(n_layers):
        p = f"encoder.layers.{i}."
        yield p + "norm_feed_forward1.weight", (D_MODEL,), ("g", 0)
        yield p + "norm_feed_forward1.bias", (D_MODEL,), ("b", 0)
        yield p + "feed_forward1.linear1.weight", (D_FF, D_MODEL), ("w", D_MODEL)
        yield p + "feed_forward1.linear2.weight", (D_MODEL, D_FF), ("wbr", D_FF)
        yield p + "norm_self_att.weight", (D_MODEL,), ("g", 0)
        yield p + "norm_self_att.bias", (D_MODEL,), ("b", 0)
        yield p + "self_attn.linear_q.weight", (D_MODEL, D_MODEL), ("w", D_MODEL)
        yield p + "self_attn.linear_k.weight", (D_MODEL, D_MODEL), ("w", D_MODEL)
        yield p + "self_attn.linear_v.weight", (D_MODEL, D_MODEL), ("w", D_MODEL)
        yield p + "self_attn.linear_pos.weight", (D_MODEL, D_MODEL), ("w", D_MODEL)
        yield p + "self_attn.linear_out.weight", (D_MODEL, D_MODEL), ("wbr", D_MODEL)
        yield p + "self_attn.pos_bias_u", (N_HEADS, D_HEAD), ("b", 0)
        yield p + "self_attn.pos_bias_v", (N_HEADS, D_HEAD), ("b", 0)
        yield p + "norm_conv.weight", (D_MODEL,), ("g", 0)
        yield p + "norm_conv.bias", (D_MODEL,), ("b", 0)
        yield p + "conv.pointwise_conv1.weight", (2 * D_MODEL, D_MODEL, 1), ("w", D_MODEL)
        yield p + "conv.depthwise_conv.weight", (D_MODEL, 1, KSIZE), ("w", KSIZE)
        yield p + "conv.batch_norm.weight", (D_MODEL,), ("g", 0)
        yield p + "conv.batch_norm.bias", (D_MODEL,), ("b", 0)
        yield p + "conv.pointwise_conv2.weight", (D_MODEL, D_MODEL, 1), ("wbr", D_MODEL)
        yield p + "norm_feed_forward2.weight", (D_MODEL,), ("g", 0)
        yield p + "norm_feed_forward2.bias", (D_MODEL,), ("b", 0)
        yield p + "feed_forward2.linear1.weight", (D_FF, D_MODEL), ("w", D_MODEL)
        yield p + "feed_forward2.linear2.weight", (D_MODEL, D_FF), ("wbr", D_FF)
        yield p + "norm_out.weight", (D_MODEL,), ("g", 0)
        yield p + "norm_out.bias", (D_MODEL,), ("b", 0)
    d = "decoder.prediction."
    yield d + "embed.weight", (VOCAB, HID), ("embed", 0)
    for l in range(2):
        yield d + f"dec_rnn.lstm.weight_ih_l{l}", (4 * HID, HID), ("w", HID)
        yield d + f"dec_rnn.lstm.weight_hh_l{l}", (4 * HID, HID), ("w", HID)
        yield d + f"dec_rnn.lstm.bias_ih_l{l}", (4 * HID,), ("b", 0)
        yield d + f"dec_rnn.lstm.bias_hh_l{l}", (4 * HID,), ("b", 0)
    yield "joint.enc.weight", (JOINT, D_MODEL), ("wenc", D_MODEL)
    yield "joint.enc.bias", (JOINT,), ("benc", n_layers)
    yield "joint.pred.weight", (JOINT, HID), ("wpred", HID)
    yield "joint.pred.bias", (JOINT,), ("b", 0)
    yield "joint.joint_net.2.weight", (VOCAB, JOINT), ("wout", JOINT)
    yield "joint.joint_net.2.bias", (VOCAB,), ("bout", 0)
    yield "preprocessor.featurizer.fb", (1, N_MELS, N_BINS), ("fb", 0)
    yield "preprocessor.featurizer.window", (WIN,), ("window", 0)


def mel_filterbank() -> np.ndarray:
    """128 x 257 triangular filters on a mel-like axis, area-normalised (data, not code)."""
    def hz_to_mel(f):
        return 2595.0 * np.log10(1.0 + f / 700.0)

    def mel_to_hz(m):
        return 700.0 * (10.0 ** (m / 2595.0) - 1.0)

    fft_freqs = np.linspace(0.0, 8000.0, N_BINS)
    pts = mel_to_hz(np.linspace(hz_to_mel(0.0), hz_to_mel(8000.0), N_MELS + 2))
    fb = np.zeros((N_MELS, N_BINS), dtype=np.float64)
    for m in range(N_MELS):
        lo, ce, hi = pts[m], pts[m + 1], pts[m + 2]
        up = (fft_freqs - lo) / max(ce - lo, 1e-9)
        dn = (hi - fft_freqs) / max(hi - ce, 1e-9)
        fb[m] = np.maximum(0.0, np.minimum(up, dn)) * (2.0 / (hi - lo))
    return fb.astype(np.float32)


def load_calibration(seed: int, n_layers: int, R, profile: str = "parity"):
    """(mu [1024] or None, blank_bias) for a (seed, n_layers, right_context) model; see tools/calibrate.py.
    profile "parity": 25 % of the frames start an emission (dense decisions for the parity tests);
    profile "speech": blank bias raised until the token rate is that of speech (~4.5 tokens per audio second) -- the bench
    workload; falls back to the parity value (with a note on stderr) where no speech calibration is committed."""
    if R is not None:
        path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "calib", f"cal_s{seed}_L{n_layers}_R{R}.npz")
        if os.path.exists(path):
            z = np.load(path)
            bb = float(z["blank_bias"])
            if profile == "speech":
                if "blank_bias_speech" in z.files:
                    bb = float(z["blank_bias_speech"])
                else:
                    import sys
                    print(f"synth: no speech-rate calibration for L={n_layers} R={R}; using the parity blank bias", file=sys.stderr)
            return z["mu"].astype(np.float32), bb
    return None, 2.8


def has_speech_calibration(seed: int, n_layers: int, R) -> bool:
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "calib", f"cal_s{seed}_L{n_layers}_R{R}.npz")
    return os.path.exists(path) and "blank_bias_speech" in np.load(path).files


_CAL_MU = None   # set by write_gguf / write_nemo_bin while generating


def gen_tensor(name: str, shape, kind, seed: int, blank_bias: float, logit_gain: float) -> np.ndarray:
    k, fan_in = kind
    rng = np.random.default_rng([seed, zlib.crc32(name.encode())])
    if k == "w":
        return (rng.standard_normal(shape, dtype=np.float32) * np.float32(1.0 / np.sqrt(fan_in)))
    if k == "wbr":       # last matrix of every residual branch: small gain keeps the random net close to identity,
        # otherwise 24 random layers collapse all frames onto one direction and the output ignores the audio
        return (rng.standard_normal(shape, dtype=np.float32) * np.float32(BRANCH_GAIN / np.sqrt(fan_in)))
    if k == "w0":        # zero-mean 3x3 filters: reject the large DC level of log-mel so frames differ
        w = rng.standard_normal(shape, dtype=np.float32)
        w -= w.mean(axis=(2, 3), keepdims=True)
        return (w * np.float32(1.0 / np.sqrt(fan_in))).astype(np.float32)
    if k == "wenc":      # encoder frames should drive the joint decision more than the prediction net
        return (rng.standard_normal(shape, dtype=np.float32) * np.float32(ENC_GAIN / np.sqrt(fan_in)))
    if k == "benc":
        # Random-weight conformers map every frame to almost the same direction (frame-to-frame
        # correlation ~0.95), which would make the RNN-T decisions ignore the audio. Cancel the
        # common component mu (per latency mode; tools/calibrate.py, committed under tools/calib/) through the bias so
        # that the joint sees the per-frame variation: b = 0.1*N - W_enc @ mu.
        b = (0.1 * rng.standard_normal(shape, dtype=np.float32)).astype(np.float32)
        if _CAL_MU is not None:
            w = gen_tensor("joint.enc.weight", (JOINT, D_MODEL), ("wenc", D_MODEL), seed, blank_bias, logit_gain)
            b = (b - w @ _CAL_MU).astype(np.float32)
        return b
    if k == "wpred":
        return (rng.standard_normal(shape, dtype=np.float32) * np.float32(PRED_GAIN / np.sqrt(fan_in)))
    if k == "g":
        return (1.0 + 0.1 * rng.standard_normal(shape, dtype=np.float32)).astype(np.float32)
    if k == "b":
        return (0.1 * rng.standard_normal(shape, dtype=np.float32)).astype(np.float32)
    if k == "embed":
        e = rng.standard_normal(shape, dtype=np.float32)
        e[VOCAB - 1] = 0.0  # blank row = padding row
        return e
    if k == "wout":
        return (rng.standard_normal(shape, dtype=np.float32) * np.float32(logit_gain / np.sqrt(fan_in)))
    if k == "bout":
        b = (0.1 * rng.standard_normal(shape, dtype=np.float32)).astype(np.float32)
        b[VOCAB - 1] += np.float32(blank_bias)
        return b
    if k == "fb":
        return mel_filterbank().reshape(shape)
    if k == "window":
        n = np.arange(WIN, dtype=np.float64)
        return (0.5 - 0.5 * np.cos(2.0 * np.pi * n / (WIN - 1))).astype(np.float32)  # symmetric Hann
    raise ValueError(k)


def make_vocab(seed: int) -> bytes:
    """1025 x 8-byte NUL-padded pieces (last = blank, empty). ~1/3 start with U+2581."""
    rng = np.random.default_rng([seed, 777])
    out = bytearray(VOCAB * 8)
    letters = "abcdefghijklmnopqrstuvwxyz"
    for i in range(VOCAB - 1):
        n = int(rng.integers(1, 5))
        body = "".join(letters[int(j)] for j in rng.integers(0, 26, n))
        piece = ("▁" + body) if rng.random() < 0.34 else body
        enc = piece.encode("utf-8")
        assert len(enc) <= 7
        out[i * 8:i * 8 + len(enc)] = enc
    return bytes(out)


# --------------------------------------------------------------------------------------
# quantisers (converter semantics)
# --------------------------------------------------------------------------------------
def quantize_q8_0(data: np.ndarray) -> bytes:
    """fp16 d = amax/127; q = round_half_even(x / fp16(d)) (convert_to_gguf.py:113-120)."""
    flat = np.ascontiguousarray(data, dtype=np.float32).reshape(-1, 32)
    amax = np.max(np.abs(flat), axis=1)
    scales = np.where(amax != 0, amax / 127.0, 0.0).astype(np.float16)
    sf = scales.astype(np.float32)[:, None]
    safe = np.where(sf != 0, sf, 1.0)
    q = np.round(flat / safe)
    q = np.where(sf != 0, q, 0).astype(np.int8)
    blk = np.empty(flat.shape[0], dtype=np.dtype([("d", np.float16), ("q", np.int8, 32)]))
    blk["d"] = scales
    blk["q"] = q
    return blk.tobytes()


def quantize_q4_0(data: np.ndarray) -> bytes:
    """Q4_0 block = fp16 d + 16 bytes of nibbles (convert_to_gguf.py:132-179): d = amax/7, q = clip(round(x / fp16(d)), -8, 7) + 8;
    byte i of a block holds element i in its low nibble and element i + 16 in its high nibble."""
    flat = np.ascontiguousarray(data, dtype=np.float32).reshape(-1, 32)
    amax = np.max(np.abs(flat), axis=1)
    scales = np.where(amax != 0, amax / 7.0, 0.0).astype(np.float16)
    sf = scales.astype(np.float32)[:, None]
    safe = np.where(sf != 0, sf, 1.0)
    q = np.clip(np.round(flat / safe), -8, 7)
    q = (np.where(sf != 0, q, 0) + 8).astype(np.uint8)
    blk = np.empty(flat.shape[0], dtype=np.dtype([("d", np.float16), ("q", np.uint8, 16)]))
    blk["d"] = scales
    blk["q"] = (q[:, :16] & 0x0F) | (q[:, 16:] << 4)
    return blk.tobytes()


def gguf_prepare(name: str, data: np.ndarray, wtype: str):
    """Apply the converter's reshape + quantise decision. Returns (dims_reversed, ggml_type, bytes)."""
    if PW_RE.search(name) and data.ndim == 3:
        data = data.squeeze(axis=2)
    elif DW_RE.search(name) and data.ndim == 3:
        data = np.ascontiguousarray(data.squeeze(axis=1).T)
    dims = list(reversed(data.shape))
    do_q = (wtype != "f32" and QUANT_RE.search(name) is not None and not DW_RE.search(name)
            and data.size >= 256 and data.ndim >= 2)
    if do_q and wtype == "f16":
        return dims, GGML_F16, data.astype(np.float16).tobytes()
    if do_q and wtype == "q8_0":
        return dims, GGML_Q8_0, quantize_q8_0(data)
    if do_q and wtype == "q4_0":
        return dims, GGML_Q4_0, quantize_q4_0(data)
    return dims, GGML_F32, np.ascontiguousarray(data, dtype=np.float32).tobytes()


def _wstr(f, s):
    b = s.encode("utf-8") if isinstance(s, str) else s
    f.write(struct.pack("<Q", len(b)))
    f.write(b)


VARIANT_TENSORS = ("joint.enc.bias", "joint.joint_net.2.bias")   # the only tensors that depend on (R, profile): calibration mean, blank bias


def _gguf_header(n_layers: int, wtype: str, seed: int):
    """(header bytes incl. alignment padding, [(name, dims, type, offset in the data section, nbytes)]) of a synthetic file."""
    import io
    specs = list(tensor_specs(n_layers))
    hparams = [("nemo.n_mels", N_MELS), ("nemo.d_model", D_MODEL), ("nemo.n_heads", N_HEADS),
               ("nemo.d_head", D_HEAD), ("nemo.d_ff", D_FF), ("nemo.n_layers", n_layers),
               ("nemo.kernel_size", 31), ("nemo.vocab_size", VOCAB), ("nemo.decoder_dim", 320),
               ("nemo.joint_dim", JOINT)]  # kernel_size=31 / decoder_dim=320 are the converter's (ignored) values
    infos, off = [], 0
    for name, shape, kind in specs:
        dims, ttype, nbytes = _prepared_size(name, shape, wtype)
        aligned = (off + ALIGN - 1) // ALIGN * ALIGN
        infos.append((name, dims, ttype, aligned, nbytes))
        off = aligned + nbytes
    f = io.BytesIO()
    f.write(GGUF_MAGIC)
    f.write(struct.pack("<I", GGUF_VERSION))
    f.write(struct.pack("<q", len(infos)))
    f.write(struct.pack("<q", len(hparams) + 3))
    for k, v in (("general.architecture", "nemo"), ("general.name", "nemotron-speech-streaming-en-0.6b"),
                 ("tokenizer.vocab", make_vocab(seed))):
        _wstr(f, k)
        f.write(struct.pack("<i", T_STR))
        _wstr(f, v)
    for k, v in hparams:
        _wstr(f, k)
        f.write(struct.pack("<i", T_U32))
        f.write(struct.pack("<I", v))
    for name, dims, ttype, aligned, _ in infos:
        _wstr(f, name)
        f.write(struct.pack("<I", len(dims)))
        for d in dims:
            f.write(struct.pack("<q", d))
        f.write(struct.pack("<i", ttype))
        f.write(struct.pack("<Q", aligned))
    pos = f.tell()
    f.write(b"\x00" * ((pos + ALIGN - 1) // ALIGN * ALIGN - pos))
    return f.getvalue(), infos


def write_gguf(path: str, n_layers: int = 24, wtype: str = "f32", seed: int = 1234,
               blank_bias: float | None = None, logit_gain: float = 1.0, R=None, mu=None, profile: str = "parity") -> None:
    """R selects the committed calibration (mean encoder output + blank bias) of that latency mode. Tensors are generated on a
    thread pool (per-tensor seeds: order-independent) and written in file order."""
    global _CAL_MU
    from concurrent.futures import ThreadPoolExecutor
    cal_mu, cal_bb = load_calibration(seed, n_layers, R, profile)
    _CAL_MU = mu if mu is not None else cal_mu
    blank_bias = cal_bb if blank_bias is None else blank_bias
    specs = list(tensor_specs(n_layers))
    header, infos = _gguf_header(n_layers, wtype, seed)

    def make(i):
        name, shape, kind = specs[i]
        _, ttype2, raw = gguf_prepare(name, gen_tensor(name, shape, kind, seed, blank_bias, logit_gain), wtype)
        assert ttype2 == infos[i][2] and len(raw) == infos[i][4], name
        return raw

    workers = max(1, min(16, len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)))
    tmp = path + f".tmp{os.getpid()}"
    with open(tmp, "wb") as f, ThreadPoolExecutor(workers) as ex:
        f.write(header)
        data_start = f.tell()
        pending, nxt, depth = {}, 0, 4 * workers                     # bounded look-ahead: at most `depth` tensors in memory
        for i in range(len(specs)):
            while nxt < len(specs) and nxt < i + depth:
                pending[nxt] = ex.submit(make, nxt); nxt += 1
            raw = pending.pop(i).result()
            cur = f.tell()
            f.write(b"\x00" * (data_start + infos[i][3] - cur))
            f.write(raw)
    os.replace(tmp, path)


def derive_gguf_variant(src: str, dst: str, n_layers: int, wtype: str, seed: int, R, profile: str) -> None:
    """Same (seed, layers, type), another latency mode / token-rate profile: only VARIANT_TENSORS differ (both stored F32), so copy the
    file and rewrite those two in place instead of regenerating 0.6 G parameters."""
    global _CAL_MU
    import shutil
    _CAL_MU, blank_bias = load_calibration(seed, n_layers, R, profile)
    header, infos = _gguf_header(n_layers, wtype, seed)
    specs = {name: (shape, kind) for name, shape, kind in tensor_specs(n_layers)}
    tmp = dst + f".tmp{os.getpid()}"
    shutil.copyfile(src, tmp)
    with open(tmp, "r+b") as f:
        assert f.read(len(header)) == header, "derive_gguf_variant: source layout differs"
        for name, dims, ttype, aligned, nbytes in infos:
            if name in VARIANT_TENSORS:
                shape, kind = specs[name]
                _, t2, raw = gguf_prepare(name, gen_tensor(name, shape, kind, seed, blank_bias, 1.0), wtype)
                assert t2 == ttype == GGML_F32 and len(raw) == nbytes, name
                f.seek(len(header) + aligned)
                f.write(raw)
    os.replace(tmp, dst)


def _prepared_size(name, shape, wtype):
    if PW_RE.search(name) and len(shape) == 3:
        shape = shape[:2]
    elif DW_RE.search(name) and len(shape) == 3:
        shape = (shape[2], shape[0])
    n = int(np.prod(shape))
    dims = list(reversed(shape))
    do_q = (wtype != "f32" and QUANT_RE.search(name) is not None and not DW_RE.search(name)
            and n >= 256 and len(shape) >= 2)
    if do_q and wtype == "f16":
        return dims, GGML_F16, n * 2
    if do_q and wtype == "q8_0":
        return dims, GGML_Q8_0, n // 32 * 34
    if do_q and wtype == "q4_0":
        return dims, GGML_Q4_0, n // 32 * 18
    return dims, GGML_F32, n * 4


def write_nemo_bin(path: str, n_layers: int = 24, seed: int = 1234,
                   blank_bias: float | None = None, logit_gain: float = 1.0, R=None) -> None:
    global _CAL_MU
    _CAL_MU, cal_bb = load_calibration(seed, n_layers, R)
    blank_bias = cal_bb if blank_bias is None else blank_bias
    specs = list(tensor_specs(n_layers))
    tmp = path + ".tmp"
    with open(tmp, "wb") as f:
        f.write(b"NEMO")
        f.write(struct.pack("<I", 1))
        f.write(struct.pack("<I", len(specs)))
        for name, shape, kind in specs:
            t = gen_tensor(name, shape, kind, seed, blank_bias, logit_gain)
            nb = name.encode()
            f.write(struct.pack("<I", len(nb)))
            f.write(nb)
            f.write(struct.pack("<I", len(shape)))
            for d in shape:
                f.write(struct.pack("<I", d))
            f.write(struct.pack("<I", 0))
            f.write(np.ascontiguousarray(t, dtype=np.float32).tobytes())
    os.replace(tmp, path)


# --------------------------------------------------------------------------------------
# audio
# --------------------------------------------------------------------------------------
def synth_pcm(stream: int, seconds: float, sr: int = 16000) -> np.ndarray:
    """Seeded, non-stationary s16 audio: a sequence of 60-320 ms 'phone-like' segments, each a sum
    of 3 sines (100-3000 Hz, random amplitudes) or a silence, over N(0, 0.02) noise; +-0.5 FS peak.
    Non-stationarity matters: it makes encoder frames (and therefore RNN-T decisions) vary in time."""
    rng = np.random.default_rng(1000 + stream)
    n = int(round(seconds * sr))
    x = np.zeros(n)
    pos = 0
    while pos < n:
        seg = int(rng.uniform(0.06, 0.32) * sr)
        end = min(n, pos + seg)
        t = np.arange(end - pos, dtype=np.float64) / sr
        if rng.random() > 0.15:                      # 15 % of segments are silence
            amp = rng.uniform(0.2, 1.0)
            for _ in range(3):
                f = rng.uniform(100.0, 3000.0)
                x[pos:end] += amp * rng.uniform(0.3, 1.0) * np.sin(2 * np.pi * f * t + rng.uniform(0, 2 * np.pi))
            ramp = np.minimum(1.0, np.minimum(t, t[::-1]) / 0.005)   # 5 ms fade to avoid clicks
            x[pos:end] *= ramp
        pos = end
    x = x / max(np.max(np.abs(x)), 1e-9) * 0.5 + rng.normal(0.0, 0.02, n) * 0.5
    x = np.clip(x, -1.0, 1.0)
    return np.round(x * 32767.0).astype(np.int16)


def sine_pcm(seconds: float, freq: float = 440.0, sr: int = 16000) -> np.ndarray:
    """The reference's own smoke input (tests/test_streaming.cpp:745-755)."""
    n = int(seconds * sr)
    t = np.arange(n, dtype=np.float32) / np.float32(sr)
    return (np.float32(0.5) * np.sin(np.float32(2.0 * np.pi * freq) * t) * np.float32(32767.0)).astype(np.int16)


def cached_model(kind: str, n_layers: int, seed: int = 1234, cache_dir: str | None = None, R: int | None = 1,
                 profile: str = "parity") -> str:
    """Materialise (once) and return the path of a synthetic model file. kind: f32|f16|q8_0|q4_0|nemo.
    R = latency mode whose calibration (tools/calib/) shapes joint.enc.bias and the blank bias;
    profile = "parity" (tests) | "speech" (bench: speech-like token rate, see load_calibration)."""
    # per user: a directory another user created first would not be writable
    cache_dir = cache_dir or os.environ.get("NSB_SYNTH_DIR") or os.path.join(tempfile.gettempdir(), f"nsb200_synth_{os.getuid()}")
    os.makedirs(cache_dir, exist_ok=True)
    ext = "bin" if kind == "nemo" else "gguf"
    tag = "" if profile == "parity" else f"_{profile}"
    path = os.path.join(cache_dir, f"synth_s{seed}_L{n_layers}_R{R}{tag}_{kind}.{ext}")
    if not os.path.exists(path):
        if kind == "nemo":
            if profile != "parity":
                raise ValueError("NEMO bins are written with the parity calibration only")
            write_nemo_bin(path, n_layers, seed, R=R)
        else:
            import glob
            sibs = sorted(glob.glob(os.path.join(cache_dir, f"synth_s{seed}_L{n_layers}_R*_{kind}.gguf")))
            if sibs:
                derive_gguf_variant(sibs[0], path, n_layers, kind, seed, R, profile)
            else:
                write_gguf(path, n_layers, kind, seed, R=R, profile=profile)
    return path


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out")
    ap.add_argument("--type", default="f32", choices=["f32", "f16", "q8_0", "q4_0", "nemo"])
    ap.add_argument("--layers", type=int, default=24)
    ap.add_argument("--seed", type=int, default=1234)
    ap.add_argument("--right-context", type=int, default=1)
    a = ap.parse_args()
    if a.type == "nemo":
        write_nemo_bin(a.out, a.layers, a.seed, R=a.right_context)
    else:
        write_gguf(a.out, a.layers, a.type, a.seed, R=a.right_context)
    print(a.out, os.path.getsize(a.out))


if __name__ == "__main__":
    main()
