"""Operator tests of the step's GEMM launches and of the split-K fold in its LayerNorm kernels, against float64 (nsb_op_gemm_ex /
nsb_op_layernorm, include/nsb200.h).

The end-to-end tests compare the encoder output within the noise of 16-bit activations (1e-3 .. 3e-2); a GEMM can be wrong by one
k-block, one row or one tile of columns inside that band. Here every launch the step makes -- each weight kind at batch sizes on both
sides of every dispatch threshold, every forced tile config, every epilogue (bias, ReLU, SiLU to f32 / f16 / bf16, residual, split-K
planes with and without C0, the output row map of the stem projection) and the 3xTF32 path of the matrices kept in F32 -- is compared
with a float64 product of the operand values the kernel actually multiplies:
  * activations rounded to the engine's activation type (round to nearest even); F32 matrices take plain fp32 activations;
  * F16 weights as stored, rounded to bf16 in BF16 mode; Q8_0 / Q4_0 weights as fp16(fp16(d) * q) (the dequantisation kernels
    multiply with __hmul2: one rounding of the exact product);
  * 3xTF32: the plain fp32 operands (the split into tf32 hi / lo parts is what is being tested), except for split-K planes, which are
    compared per plane against the [hi | hi | lo] x [hi | lo | hi] operands of their own k range.
Metric, per element: r = (|y - y64| - half an ulp of a 16-bit output) / (|x| @ |W|^T + |bias| + tiny). It does not depend on scale;
skipping one k-block moves it to ~5e-2, far above fp32 accumulation noise (~1e-6). Every destination is surrounded by guard rows
and columns holding a NaN pattern (the live region too, so an element the kernel does not write stays NaN): the op counts changed guard
elements, which must be 0. With NSB_GEMM_OPS_REPORT=<file> set, the measured maximum of every case is appended to that file as one
JSON line: the data the bounds below are set from.
"""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TINY = 1e-30
MAX_ROWS = 1792

# Bounds on r (module docstring), each 2x - 3.5x above the largest value measured over every case of its class on an NVIDIA B200
# (1000 W power limit). A GEMM that skips one k-block measures 6e-2 - 8e-2; bias added to every split-K slice, 10.
BOUND_16 = 3e-6          # fp16 / bf16 / Q8_0 / Q4_0 operands, fp32 accumulation: measured 8.5e-7 (ff1b, K = 4096), 1.4e-6 with the residual epilogue
# 3xTF32 against plain fp32 operands: measured 6.1e-6 (stem projection, K = 4352). Mostly the tensor cores' fp32 accumulation, not the
# split: a split-K plane against its own exact tf32 hi / lo operands alone measures up to 3.2e-6. Single-pass tf32 measures 1.3e-4.
BOUND_TF32X3 = 2e-5
BOUND_SIMT = 2.0 ** -20  # SIMT fp32: measured 3.9e-7
BOUND_LN = 1e-6          # LayerNorm, relative to |g| (|z| + 1), beyond half an ulp of a 16-bit output: measured 3.3e-7
# the same with a common offset of 1e3: measured 1.6e-4, the fp32 rounding of the reduced rows (ulp(1e3) / 2 = 3e-5) and of the fp32
# row sums; a one-pass E[x^2] - E[x]^2 in fp32 would keep ~4 bits of the variance (E[x^2] = 1e6 against a variance of 1)
BOUND_LN_OFFSET = 4e-4

GGML_F32, GGML_F16, GGML_Q4_0, GGML_Q8_0 = 0, 1, 2, 8
L1 = "encoder.layers.1."
# name, (n_out, n_in), tensors it is stacked from
WEIGHTS = {
    "ff1a": (L1 + "feed_forward1.linear1.weight", None),
    "ff1b": (L1 + "feed_forward1.linear2.weight", None),
    "qkv": (L1 + "self_attn.linear_qkv.weight", [L1 + f"self_attn.linear_{c}.weight" for c in "qkv"]),
    "out": (L1 + "self_attn.linear_out.weight", None),
    "pw1": (L1 + "conv.pointwise_conv1.weight", None),
    "pw2": (L1 + "conv.pointwise_conv2.weight", None),
    "conv3": ("encoder.pre_encode.conv.3.weight", None),
    "conv6": ("encoder.pre_encode.conv.6.weight", None),
    "stem_out": ("encoder.pre_encode.out.weight", None),
    "joint_enc": ("joint.enc.weight", None),
}
SHAPES = {"ff1a": (4096, 1024), "ff1b": (1024, 4096), "qkv": (3072, 1024), "out": (1024, 1024), "pw1": (2048, 1024), "pw2": (1024, 1024),
          "conv3": (256, 256), "conv6": (256, 256), "stem_out": (1024, 4352), "joint_enc": (640, 1024)}
F32_KINDS = ("conv3", "conv6", "stem_out", "joint_enc")


# ------------------------------------------------------------------------------------------------------------------------------
# host reconstruction of the kernel's operands (CPU, pinned by the unmarked tests below)
# ------------------------------------------------------------------------------------------------------------------------------
def round_bf16(a):
    """fp32 -> bf16 -> fp32, round to nearest even (finite inputs)."""
    u = np.ascontiguousarray(a, dtype=np.float32).view(np.uint32).astype(np.uint64)
    u = ((u + 0x7FFF + ((u >> 16) & 1)) >> 16) << 16
    return u.astype(np.uint32).view(np.float32)


def round_f16(a):
    return np.asarray(a, dtype=np.float32).astype(np.float16).astype(np.float32)


def to_tf32(a):
    """cvt.rna.tf32.f32: 10 mantissa bits, round to nearest, ties away from zero (finite inputs)."""
    u = np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)
    return ((u + np.uint32(0x1000)) & np.uint32(0xFFFFE000)).view(np.float32)


def split_tf32(a):
    hi = to_tf32(a)
    return hi, to_tf32(np.asarray(a, dtype=np.float32) - hi)


def decode16(bits, out_type):
    import nsb200
    if out_type == nsb200.OUT_F16:
        return bits.view(np.float16).astype(np.float64)
    return (bits.astype(np.uint32) << 16).view(np.float32).astype(np.float64)


def half_ulp(v, out_type):
    """half an ulp of the 16-bit output type at |v| (normal range; subnormals at the smallest normal spacing)."""
    import nsb200
    mant, emin = (10, -14) if out_type == nsb200.OUT_F16 else (7, -126)
    e = np.floor(np.log2(np.maximum(np.abs(v), 2.0 ** emin)))
    return 2.0 ** (np.maximum(e, emin) - mant - 1)


def act_operand(x, act):
    """what the engine multiplies for activations x: act = 'f16' / 'bf16' (rounded) or 'f32' (plain)."""
    return round_f16(x) if act == "f16" else round_bf16(x) if act == "bf16" else np.asarray(x, dtype=np.float32)


def read_matrix(path, kind):
    import nsb200
    name, parts = WEIGHTS[kind]
    n_out, n_in = SHAPES[kind]
    mats, types = [], set()
    for p in parts or [name]:
        w, t = nsb200.read_tensor(path, p)
        mats.append(w.reshape(-1, n_in)); types.add(t)
    w = np.concatenate(mats, axis=0)
    if kind == "stem_out":                          # the engine's NHWC flattening: column (x * 256 + c) holds the file's (c * 17 + x)
        w = np.ascontiguousarray(w.reshape(n_out, 256, 17).transpose(0, 2, 1).reshape(n_out, n_in))
    assert w.shape == (n_out, n_in) and len(types) == 1
    return w, types.pop()


def weight_operand(w, ggml_type, mode):
    """the weight values the kernel multiplies in engine mode 'f16' / 'bf16' / 'q8' / 'f32' (F32 matrices: plain fp32)."""
    if ggml_type in (GGML_Q8_0, GGML_Q4_0):
        return round_f16(w)                         # fp16(d) * q in f32 is exact; __hmul2 rounds it once to fp16
    if mode == "bf16":
        return round_bf16(w)
    if mode == "f16" and ggml_type == GGML_F32:
        return round_f16(w)
    return np.asarray(w, dtype=np.float32)


# ------------------------------------------------------------------------------------------------------------------------------
# CPU tests of the helpers
# ------------------------------------------------------------------------------------------------------------------------------
def test_bf16_rounding_matches_torch():
    import torch
    rng = np.random.default_rng(0)
    x = np.concatenate([(rng.standard_normal(100000) * 10.0 ** rng.integers(-30, 30, 100000)).astype(np.float32),
                        # exact ties (low 16 bits 0x8000) with both parities of the kept bit
                        (np.arange(1000, dtype=np.uint32) << 16 | 0x3F800000 | 0x8000).view(np.float32)])
    ref = torch.from_numpy(x).to(torch.bfloat16).to(torch.float32).numpy()
    assert np.array_equal(round_bf16(x), ref)


def test_tf32_split_is_exact_and_rounds_ties_away():
    rng = np.random.default_rng(1)
    x = rng.standard_normal(100000).astype(np.float32)
    hi, lo = split_tf32(x)
    for p in (hi, lo):
        assert not (p.view(np.uint32) & 0x1FFF).any()                        # representable in tf32
    assert np.all(np.abs((hi.astype(np.float64) + lo) - x) <= np.abs(x) * 2.0 ** -21)
    tie = np.array([0x3F801000, 0xBF801000], dtype=np.uint32).view(np.float32)   # 1 + 2^-11 (a tie), and its negative
    assert np.array_equal(to_tf32(tie), np.array([0x3F802000, 0xBF802000], dtype=np.uint32).view(np.float32))


def _block_bytes(path, name, n_bytes):
    """raw bytes of a tensor of the synthetic GGUF: its offset from the tensor info, the data section located through an F32 tensor"""
    import struct
    import nsb200
    raw = open(path, "rb").read()

    def info(n):
        at = raw.index(struct.pack("<Q", len(n)) + n.encode()) + 8 + len(n)
        nd = struct.unpack_from("<I", raw, at)[0]
        return struct.unpack_from("<IQ", raw, at + 4 + 8 * nd)              # type, offset in the data section
    probe = "encoder.pre_encode.conv.0.bias"
    v, t = nsb200.read_tensor(path, probe)
    assert t == GGML_F32
    data = raw.index(v.tobytes()) - info(probe)[1]
    t, off = info(name)
    return t, raw[data + off:data + off + n_bytes]


@pytest.mark.parametrize("wtype", ["q8_0", "q4_0"])
def test_quantised_weight_operand_matches_block_bytes(built, wtype):
    """weight_operand() of a Q8_0 / Q4_0 matrix == fp16(fp16(d) * q) decoded straight from the blocks of the file"""
    path = synth.cached_model(wtype, 2, R=0)
    kind = "pw1"
    w, t = read_matrix(path, kind)
    n = w.size
    bs = 34 if wtype == "q8_0" else 18
    t2, raw = _block_bytes(path, WEIGHTS[kind][0], n // 32 * bs)
    assert t == t2 == (GGML_Q8_0 if wtype == "q8_0" else GGML_Q4_0)
    blk = np.frombuffer(raw, dtype=np.uint8).reshape(-1, bs)
    d = blk[:, :2].copy().view(np.float16).astype(np.float32)            # [nb, 1]
    if wtype == "q8_0":
        q = blk[:, 2:].view(np.int8).astype(np.float32)
    else:
        nib = blk[:, 2:]
        q = np.concatenate([nib & 0x0F, nib >> 4], axis=1).astype(np.float32) - 8.0   # element i: low nibble of byte i, i + 16: high
    ref = (d * q).astype(np.float16).astype(np.float32).reshape(w.shape)
    got = weight_operand(w, t, "q8")
    assert np.array_equal(got, ref)
    assert np.abs(got).max() > 0


# ------------------------------------------------------------------------------------------------------------------------------
# GPU side: engines, float64 products, ratios
# ------------------------------------------------------------------------------------------------------------------------------
def report(**kw):
    path = os.environ.get("NSB_GEMM_OPS_REPORT")
    if path:
        with open(path, "a") as f:
            f.write(json.dumps(kw) + "\n")


# engine mode -> (GGUF weight type, compute, activation operand type)
MODES = {"f16": ("f16", 2, "f16"), "bf16": ("f16", 3, "bf16"), "q8_0": ("q8_0", 0, "f16"), "q4_0": ("q4_0", 0, "f16"), "f32": ("f32", 1, "f32")}
_engines = {}


@pytest.fixture(scope="module")
def engines(built):
    yield _engine
    for e in _engines.values():
        e.close()
    _engines.clear()
    _products.clear()


def _engine(mode):
    import nsb200
    if mode not in _engines:
        wtype, compute, _ = MODES[mode]
        _engines[mode] = nsb200.Engine(synth.cached_model(wtype, 2, R=0), right_context=0, max_streams=1, compute=compute)
    return _engines[mode]


def _x(n_in, seed=0):
    return np.random.default_rng(1000 + n_in + seed).standard_normal((MAX_ROWS, n_in)).astype(np.float32)


_products = {}


def operands(mode, kind):
    """(x operand, W operand, plain fp32 x) in float64 on the GPU for MAX_ROWS rows; row counts below use a prefix"""
    import torch
    key = ("ops", mode, kind)
    if key not in _products:
        wtype, _, act = MODES[mode]
        w, t = read_matrix(synth.cached_model(wtype, 2, R=0), kind)
        x = _x(SHAPES[kind][1])
        f32 = kind in F32_KINDS or mode == "f32"
        xo = x if f32 else act_operand(x, act)
        wo = np.asarray(w, dtype=np.float32) if f32 else weight_operand(w, t, "q8" if mode in ("q8_0", "q4_0") else mode)
        dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to("cuda", torch.float64)
        _products[key] = (dev(xo), dev(wo), x)
    return _products[key]


def product(mode, kind):
    """float64 (x W^T, |x| |W|^T) for MAX_ROWS rows, cached per (mode, weight)"""
    key = ("prod", mode, kind)
    if key not in _products:
        for k in [k for k in _products if k[0] == "prod"][:-4]:             # a handful of products stay resident
            del _products[k]
        xo, wo, _ = operands(mode, kind)
        _products[key] = (xo @ wo.T, xo.abs() @ wo.abs().T)
    return _products[key]


def bound_for(mode, kind):
    if kind in F32_KINDS and mode != "f32":
        return BOUND_TF32X3
    return BOUND_SIMT if mode == "f32" else BOUND_16


def ratio(y, y64, den, out_type=0):
    """max over elements of r (module docstring); y: what the op returned (float32, or uint16 bits), y64 / den: torch float64"""
    import torch
    import nsb200
    if out_type == nsb200.OUT_F32:
        yv = torch.from_numpy(np.ascontiguousarray(y)).to("cuda", torch.float64)
        err = (yv - y64).abs()
    else:
        yv = torch.from_numpy(decode16(y, out_type)).to("cuda")
        err = ((yv - y64).abs() - torch.from_numpy(half_ulp(y64.cpu().numpy(), out_type)).to("cuda")).clamp_min(0.0)
    r = err / (den + TINY)
    assert bool(torch.isfinite(r).all()), "non-finite output (an element the kernel did not write keeps the NaN fill)"
    return float(r.max())


def gemm(eng, kind, x, **kw):
    y, bad = eng.op_gemm_ex(WEIGHTS[kind][0], x, **kw)
    assert bad == 0, f"{bad} guard elements written"
    return y


# ---- default dispatch ------------------------------------------------------------------------------------------------------------
ROWS = [1, 7, 127, 128, 129, 255, 256, 257, 513, 900, 1024, 1025, 1792]
# variant -> (engine mode, environment): Q8_0 / Q4_0 through the fp16 expansion (default) and through the fused-dequantisation kernels
# (single-CTA tiles below 4 row tiles, 256-row pair tiles above); 16-bit with the persistent pair tiles
VARIANTS = {
    "f16": ("f16", {}), "bf16": ("bf16", {}), "f16_persist": ("f16", {"NSB_PAIR256_PERSIST": "1"}),
    "q8_0_expand": ("q8_0", {}), "q8_0_fused": ("q8_0", {"NSB_Q8_PREDEQUANT_ROWS": "1000000", "NSB_Q8_PAIR": "1"}),
    "q4_0_expand": ("q4_0", {}), "q4_0_fused": ("q4_0", {"NSB_Q8_PREDEQUANT_ROWS": "1000000", "NSB_Q8_PAIR": "1"}),
    "f32_simt": ("f32", {}),
}


def use_variant(variant, monkeypatch):
    mode, env = VARIANTS[variant]
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    return mode


@pytest.mark.gpu
@pytest.mark.parametrize("kind", list(WEIGHTS))
@pytest.mark.parametrize("variant", list(VARIANTS))
def test_default_dispatch(engines, variant, kind, monkeypatch):
    mode = use_variant(variant, monkeypatch)
    eng = engines(mode)
    _, _, x = operands(mode, kind)
    y64, den = product(mode, kind)
    bound = bound_for(mode, kind)
    worst = {}
    for rows in ROWS:
        y = gemm(eng, kind, x[:rows])
        worst[rows] = ratio(y, y64[:rows], den[:rows])
        report(test="default", variant=variant, weight=kind, rows=rows, r=worst[rows], bound=bound)
    if variant in ("f16", "q8_0_fused"):                                       # same call twice: same bits
        assert np.array_equal(gemm(eng, kind, x[:900]), gemm(eng, kind, x[:900]))
    bad = {r: v for r, v in worst.items() if not v <= bound}
    assert not bad, (bound, bad)


# ---- forced tile configs ---------------------------------------------------------------------------------------------------------
FORCED = [(32, 4), (32, 5), (32, 8), (64, 4), (64, 6), (64, 98), (128, 3), (128, 4), (256, 2), (256, 3),
          (112, 97), (160, 97), (208, 97), (256, 97), (112, 96), (128, 96), (160, 96), (208, 96), (256, 96)]
FORCED_Q8 = [(112, 95), (160, 95), (208, 95)]
TF32_TILES = {(32, 5), (64, 4), (128, 3), (128, 4), (256, 2)}
N_KIND = {256: "conv3", 640: "joint_enc", 1024: "out", 2048: "pw1", 3072: "qkv", 4096: "ff1a"}


def forced_ok(bn, st, kind, q8_planes=False):
    """whether the op must accept the forced config (the rest must raise NSB_ERR_ARG)"""
    n = SHAPES[kind][0]
    if kind in F32_KINDS:                                                      # tf32 operands
        return (bn, st) in TF32_TILES and n % bn == 0
    if q8_planes:
        return st == 95
    if st == 95:
        return False
    return st in (96, 97) or n % bn == 0


@pytest.mark.gpu
@pytest.mark.parametrize("bn,st", FORCED + FORCED_Q8, ids=[f"{b}_{s}" for b, s in FORCED + FORCED_Q8])
def test_forced_tile_configs(engines, bn, st, monkeypatch):
    import nsb200
    q8 = st == 95
    mode = "q8_0" if q8 else "f16"
    if q8:                                                                     # keep the Q8_0 planes: the fused kernels take them
        monkeypatch.setenv("NSB_Q8_PREDEQUANT_ROWS", "1000000")
    eng = engines(mode)
    for n, kind in N_KIND.items():
        _, _, x = operands(mode, kind)
        y64, den = product(mode, kind)
        for rows in (1, 129, 900):
            if not forced_ok(bn, st, kind, q8_planes=q8):
                with pytest.raises(nsb200.NsbError, match=r"nsb error -1:.*forced tile"):
                    eng.op_gemm_ex(WEIGHTS[kind][0], x[:rows], force_bn=bn, force_stages=st)
                continue
            r = ratio(gemm(eng, kind, x[:rows], force_bn=bn, force_stages=st), y64[:rows], den[:rows])
            report(test="forced", config=f"{bn}/{st}", weight=kind, n=n, rows=rows, r=r, bound=bound_for(mode, kind))
            assert r <= bound_for(mode, kind), (kind, rows, r)


@pytest.mark.gpu
def test_forced_16bit_tile_on_quantised_planes_is_refused(engines, monkeypatch):
    import nsb200
    monkeypatch.setenv("NSB_Q8_PREDEQUANT_ROWS", "1000000")
    eng = engines("q8_0")
    x = _x(1024)[:129]
    with pytest.raises(nsb200.NsbError, match=r"nsb error -1:.*Q8_0"):
        eng.op_gemm_ex(WEIGHTS["ff1a"][0], x, force_bn=64, force_stages=4)


# ---- epilogues -------------------------------------------------------------------------------------------------------------------
def _bias(n, seed=5):
    return (np.random.default_rng(seed).standard_normal(n) * 4.0).astype(np.float32)


def _twice(eng, kind, x, **kw):
    """the op twice: identical bits, no guard element touched"""
    a = gemm(eng, kind, x, **kw)
    b = gemm(eng, kind, x, **kw)
    assert np.array_equal(a, b), "two identical calls differ"
    return a


@pytest.mark.gpu
@pytest.mark.parametrize("epi", ["bias", "relu_bias", "silu"])
@pytest.mark.parametrize("out", ["f32", "f16", "bf16"])
@pytest.mark.parametrize("mode,kind", [("f16", "ff1a"), ("bf16", "ff1a"), ("f16", "pw2"), ("f16", "conv3"), ("f16", "joint_enc")])
def test_epilogue_bias_relu_silu(engines, mode, kind, epi, out):
    import torch
    import nsb200
    out_type = {"f32": nsb200.OUT_F32, "f16": nsb200.OUT_F16, "bf16": nsb200.OUT_BF16}[out]
    eng = engines(mode)
    _, _, x = operands(mode, kind)
    y64, den = product(mode, kind)
    n = SHAPES[kind][0]
    bias = _bias(n)
    bt = torch.from_numpy(bias.astype(np.float64)).to("cuda")
    worst = 0.0
    for rows in (7, 129, 900):
        kw = dict(out_type=out_type)
        acc, d = y64[:rows], den[:rows]
        if epi == "silu":
            kw["epi"] = nsb200.EPI_SILU
            ref, d = acc * torch.sigmoid(acc), 1.1 * d                         # |silu'| < 1.1
        else:
            kw["bias"] = bias
            ref, d = acc + bt, d + bt.abs()
            if epi == "relu_bias":
                kw["epi"] = nsb200.EPI_RELU
                ref = ref.clamp_min(0.0)
        y = _twice(eng, kind, x[:rows], **kw)
        assert y.dtype == (np.float32 if out == "f32" else np.uint16)
        worst = max(worst, ratio(y, ref, d, out_type))
    bound = bound_for(mode, kind)
    report(test="epilogue", mode=mode, weight=kind, epi=epi, out=out, r=worst, bound=bound)
    assert worst <= bound, worst


@pytest.mark.gpu
@pytest.mark.parametrize("alpha", [1.0, 0.5])
@pytest.mark.parametrize("variant,kind", [("f16", "ff1b"), ("bf16", "out"), ("q8_0_expand", "pw2"), ("q4_0_fused", "ff1b"), ("f16", "joint_enc")])
def test_epilogue_residual(engines, variant, kind, alpha, monkeypatch):
    import torch
    import nsb200
    mode = use_variant(variant, monkeypatch)
    eng = engines(mode)
    _, _, x = operands(mode, kind)
    y64, den = product(mode, kind)
    worst = 0.0
    for rows in (1, 129, 900):
        c = np.random.default_rng(rows).standard_normal((rows, SHAPES[kind][0])).astype(np.float32) * 8.0
        ct = torch.from_numpy(c.astype(np.float64)).to("cuda")
        y = _twice(eng, kind, x[:rows], epi=nsb200.EPI_RESID, alpha=alpha, c_init=c)
        worst = max(worst, ratio(y, ct + alpha * y64[:rows], alpha * den[:rows] + ct.abs() * 2.0 ** -23))
    bound = bound_for(mode, kind)
    report(test="residual", variant=variant, weight=kind, alpha=alpha, r=worst, bound=bound)
    assert worst <= bound, worst


def plane_refs(mode, kind, rows, splits, keep=None):
    """float64 (partial product, |x| |W|^T) of each k slice: the operands of its own k range (3xTF32: [hi | hi | lo] x [hi | lo | hi])"""
    import torch
    xo, wo, x = operands(mode, kind)
    if kind in F32_KINDS and mode != "f32":
        xh, xl = split_tf32(x[:rows])
        wh, wl = split_tf32(wo.cpu().numpy().astype(np.float32))
        dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to("cuda", torch.float64)
        xo, wo = dev(np.concatenate([xh, xh, xl], axis=1)), dev(np.concatenate([wh, wl, wh], axis=1))
    xo = xo[:rows]
    if keep is not None:
        xo = xo[torch.from_numpy(keep).to("cuda")]
    kz = xo.shape[1] // splits
    return [(xo[:, z * kz:(z + 1) * kz] @ wo[:, z * kz:(z + 1) * kz].T, xo[:, z * kz:(z + 1) * kz].abs() @ wo[:, z * kz:(z + 1) * kz].abs().T)
            for z in range(splits)]


def _check_planes(y, refs, bias):
    import torch
    bt = torch.from_numpy(bias.astype(np.float64)).to("cuda")
    worst = 0.0
    assert y.shape[0] == len(refs)
    for z, (p64, d) in enumerate(refs):
        ref, den = (p64 + bt, d + bt.abs()) if z == 0 else (p64, d)            # the bias belongs to slice 0 only
        worst = max(worst, ratio(y[z], ref, den))
    return worst


@pytest.mark.gpu
@pytest.mark.parametrize("c0", [False, True], ids=["workspace", "c0"])
@pytest.mark.parametrize("splits", [2, 4, 6, 8])
@pytest.mark.parametrize("variant,kind", [("f16", "out"), ("bf16", "ff1b"), ("q8_0_expand", "ff1b"), ("q8_0_fused", "ff1b"),
                                          ("f16", "stem_out"), ("f16", "joint_enc")])
def test_epilogue_split_k_planes(engines, variant, kind, splits, c0, monkeypatch):
    import nsb200
    mode = use_variant(variant, monkeypatch)
    eng = engines(mode)
    _, _, x = operands(mode, kind)
    bias = _bias(SHAPES[kind][0])
    nk = SHAPES[kind][1] * (3 if kind in F32_KINDS else 1) // (32 if kind in F32_KINDS else 64)
    worst = 0.0
    for rows in (1, 129, 900):
        kw = dict(epi=nsb200.EPI_PARTIAL, splits=splits, c0=c0, bias=bias)
        if nk % splits:
            with pytest.raises(nsb200.NsbError, match=r"nsb error -1:.*split-K"):
                eng.op_gemm_ex(WEIGHTS[kind][0], x[:rows], **kw)
            continue
        y = _twice(eng, kind, x[:rows], **kw)
        assert y.shape == (splits, rows, SHAPES[kind][0])
        worst = max(worst, _check_planes(y, plane_refs(mode, kind, rows, splits), bias))
    if nk % splits == 0:
        bound = bound_for(mode, kind)
        report(test="split_k", variant=variant, weight=kind, splits=splits, c0=c0, r=worst, bound=bound)
        assert worst <= bound, worst


@pytest.mark.gpu
@pytest.mark.parametrize("T", [1, 2, 7, 14])
def test_output_row_map(engines, T):
    """c_group = T + 2, c_drop = 2: the stem projection as the step runs it (all T + 2 frames of every stream in, the two pre-encode
    frames dropped, split-K planes with slice 0 + bias in C0), and a 16-bit output through the same row map"""
    import torch
    import nsb200
    g = T + 2
    worst = {}
    for B in (1, 3, 64):
        rows = B * g
        keep = np.array([r for r in range(rows) if r % g >= 2])
        m_out = B * T
        # stem projection: 3xTF32, 8 slices, C0 + bias
        eng = engines("f16")
        _, _, x = operands("f16", "stem_out")
        bias = _bias(1024)
        y = _twice(eng, "stem_out", x[:rows], epi=nsb200.EPI_PARTIAL, splits=8, c0=True, bias=bias, c_group=g, c_drop=2)
        assert y.shape == (8, m_out, 1024)
        worst["stem_out"] = max(worst.get("stem_out", 0.0), _check_planes(y, plane_refs("f16", "stem_out", rows, 8, keep), bias))
        # 16-bit outputs through the row map (single-CTA, 128-row pair and 256-row pair tiles as the row count grows)
        for mode, kind, out_type in (("bf16", "ff1a", nsb200.OUT_BF16), ("f16", "pw2", nsb200.OUT_F16)):
            y64, den = product(mode, kind)
            _, _, x = operands(mode, kind)
            y = _twice(engines(mode), kind, x[:rows], out_type=out_type, c_group=g, c_drop=2)
            assert y.shape == (m_out, SHAPES[kind][0])
            kt = torch.from_numpy(keep).to("cuda")
            worst[kind] = max(worst.get(kind, 0.0), ratio(y, y64[:rows][kt], den[:rows][kt], out_type))
    report(test="row_map", T=T, r=worst)
    bad = {k: v for k, v in worst.items() if not v <= bound_for("f16", k)}
    assert not bad, bad


@pytest.mark.gpu
@pytest.mark.parametrize("rotate", [0, 1])
def test_rotate(engines, rotate):
    eng = engines("f16")
    worst = 0.0
    for kind, force in (("ff1a", (0, 0)), ("ff1b", (64, 4)), ("out", (32, 5)), ("joint_enc", (32, 5))):
        _, _, x = operands("f16", kind)
        y64, den = product("f16", kind)
        for rows in (1, 129, 900):
            y = gemm(eng, kind, x[:rows], rotate=rotate, force_bn=force[0], force_stages=force[1])
            worst = max(worst, ratio(y, y64[:rows], den[:rows]) / bound_for("f16", kind))
    report(test="rotate", rotate=rotate, r_over_bound=worst)
    assert worst <= 1.0, worst


# ---- 3xTF32 really is three passes -----------------------------------------------------------------------------------------------
def f32_matrix_ratio():
    """max r of the F32 matrices (3xTF32 in F16 mode) at 129 rows against plain fp32 operands, computed on the host. Run in a subprocess
    with NSB_STEM_TF32=1 (single-pass tf32; read once per process) it must exceed BOUND_TF32X3."""
    import nsb200
    path = synth.cached_model("f16", 2, R=0)
    eng = nsb200.Engine(path, right_context=0, max_streams=1, compute=2)
    worst = 0.0
    for kind in F32_KINDS:
        w, _ = read_matrix(path, kind)
        x = _x(SHAPES[kind][1])[:129]
        y, bad = eng.op_gemm_ex(WEIGHTS[kind][0], x)
        assert bad == 0
        x64, w64 = x.astype(np.float64), w.astype(np.float64)
        worst = max(worst, float((np.abs(y - x64 @ w64.T) / (np.abs(x64) @ np.abs(w64).T + TINY)).max()))
    eng.close()
    return worst


@pytest.mark.gpu
def test_single_pass_tf32_fails_the_3xtf32_bound(built):
    here = f32_matrix_ratio()
    code = ("import sys; sys.path[:0] = [{!r}, {!r}, {!r}]; import test_gpu_gemm_ops as t; print(t.f32_matrix_ratio())"
            .format(os.path.join(ROOT, "tests"), ROOT, os.path.join(ROOT, "tools")))
    out = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, NSB_STEM_TF32="1"), capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    single = float(out.stdout.strip().splitlines()[-1])
    report(test="stem_tf32", r_3xtf32=here, r_single_pass=single, bound=BOUND_TF32X3)
    assert here <= BOUND_TF32X3, here
    assert single > BOUND_TF32X3, single


# ---- LayerNorm fold --------------------------------------------------------------------------------------------------------------
def ln64(x, g, b):
    m = x.mean(axis=1, keepdims=True)
    v = ((x - m) ** 2).mean(axis=1, keepdims=True)
    z = (x - m) / np.sqrt(v + 1e-5)
    return z * g + b, z


def ln_ratio(y, y64, z, g, out_type):
    import nsb200
    if out_type == nsb200.OUT_F32:
        err = np.abs(y.astype(np.float64) - y64)
    else:
        err = np.maximum(np.abs(decode16(y, out_type) - y64) - half_ulp(y64, out_type), 0.0)
    r = err / (np.abs(g) * (np.abs(z) + 1.0))
    assert np.isfinite(r).all()
    return float(r.max())


@pytest.mark.gpu
@pytest.mark.parametrize("offset", [0.0, 1e3], ids=["centred", "offset1e3"])
@pytest.mark.parametrize("kind", ["ln", "ln2", "ln2_last"])
@pytest.mark.parametrize("rows", [1, 7, 1023, 1024, 1025, 1792])
def test_layernorm_fold(engines, rows, kind, offset):
    """LayerNorm of x + alpha * (sum of split-K planes), both kernels on each side of the 1024-row switch (16-bit outputs), plain and
    fused with the next layer's first norm (ln2), and the last layer's norm_out (ln2_last: no second norm)"""
    import nsb200
    eng = engines("f16")
    rng = np.random.default_rng(rows)
    x = (offset + rng.standard_normal((rows, 1024))).astype(np.float32)
    P = (rng.standard_normal((8, rows, 1024)) * 0.5).astype(np.float32)
    g1, b1, g2, b2 = [(c + 0.2 * rng.standard_normal(1024)).astype(np.float32) for c in (1.0, 0.0, 1.0, 0.0)]
    bound = BOUND_LN_OFFSET if offset else BOUND_LN
    worst = 0.0
    for out_type in (nsb200.OUT_F32, nsb200.OUT_F16, nsb200.OUT_BF16):
        for n_planes in (0, 1, 2, 7, 8):
            for alpha in ((1.0, 0.5) if n_planes else (1.0,)):
                kw = dict(planes=P[:n_planes] if n_planes else None, alpha=alpha, out_type=out_type)
                if kind != "ln":
                    kw.update(fused=True, g2=g2 if kind == "ln2" else None, b2=b2 if kind == "ln2" else None)
                x_out, y = eng.op_layernorm(x, g1, b1, **kw)
                # the reduced rows the step relies on: x + alpha * (((0 + p0) + p1) + ...) in fp32, summed in plane order
                acc = np.zeros_like(x)
                for z in range(n_planes):
                    acc = acc + P[z]
                xr32 = x + np.float32(alpha) * acc
                xr = x.astype(np.float64) + alpha * P[:n_planes].astype(np.float64).sum(axis=0)
                y1, z1 = ln64(xr, g1.astype(np.float64), b1.astype(np.float64))
                if kind == "ln":
                    assert np.array_equal(x_out, xr32), "the reduced x written back differs"
                    worst = max(worst, ln_ratio(y, y1, z1, g1, out_type))
                else:
                    worst = max(worst, ln_ratio(x_out, y1, z1, g1, nsb200.OUT_F32))     # x <- LN1(x), f32
                    if kind == "ln2":
                        y2, z2 = ln64(x_out.astype(np.float64), g2.astype(np.float64), b2.astype(np.float64))
                        worst = max(worst, ln_ratio(y, y2, z2, g2, out_type))
                    else:
                        assert not y.any(), "norm_out of the last layer writes no second output"
    report(test="layernorm", rows=rows, kind=kind, offset=offset, r=worst, bound=bound)
    assert worst <= bound, worst


@pytest.mark.gpu
def test_layernorm_refuses_more_than_eight_planes(engines):
    import nsb200
    eng = engines("f16")
    x = np.zeros((4, 1024), np.float32)
    one = np.ones(1024, np.float32)
    with pytest.raises(nsb200.NsbError, match=r"nsb error -1:"):
        eng.op_layernorm(x, one, one, planes=np.zeros((9, 4, 1024), np.float32))
