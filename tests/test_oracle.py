"""CPU tests of the oracle (oracle/stream_oracle.cpp): pinned against
  (a) the committed golden vectors in tests/golden/ -- produced by tools/make_golden.py from the reference's OWN code
      (src/preprocessor.cpp, src/reference/*.cpp compiled into oracle/_ref/libnemo_ref.so), and
  (b) that library directly, when it is present (this container; the prebuilt .so also travels to the GPU box),
plus the structural facts SURVEY.md 8(a)/(c) derives from the reference (chunk arithmetic, shapes) and
self-consistency properties of the cache carry-over that no reference test pins."""
import os

import numpy as np
import pytest

import oracle as O
import synth

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(scope="module")
def model2(built):
    return O.Model(synth.cached_model("f32", 2, R=0))


def test_mel_matches_reference_golden_bit_exact(built):
    g = np.load(os.path.join(GOLD, "mel_ref.npz"))
    m = O.Model(synth.cached_model("f32", 2, R=0))
    pp = O.Preproc(model=m)
    mel = np.concatenate([pp.process(g["pcm"][i:i + 2720]) for i in range(0, len(g["pcm"]), 2720)])
    assert mel.shape == g["mel"].shape
    assert np.array_equal(mel.view(np.uint32), g["mel"].view(np.uint32))
    mel_sine = O.Preproc(model=m).process(g["sine"])
    assert np.array_equal(mel_sine.view(np.uint32), g["mel_sine"].view(np.uint32))


def test_mel_is_push_granularity_independent(built, model2):
    pcm = synth.synth_pcm(3, 0.8)
    whole = O.Preproc(model=model2).process(pcm)
    pp, parts, i, rng = O.Preproc(model=model2), [], 0, np.random.default_rng(1)
    while i < len(pcm):
        n = int(rng.integers(1, 700))
        parts.append(pp.process(pcm[i:i + n])); i += n
    parts = np.concatenate(parts)
    assert np.array_equal(whole.view(np.uint32), parts.view(np.uint32))
    # frame count formula of get_full_frames (src/preprocessor.cpp:320-328): (256 + n - 512 + 160) / 160
    assert whole.shape[0] == (256 + len(pcm) - 512 + 160) // 160


def test_mel_edge_cases(built, model2):
    pp = O.Preproc(model=model2)
    assert pp.process(np.zeros(0, np.int16)).shape[0] == 0          # empty push
    assert pp.process(np.zeros(255, np.int16)).shape[0] == 0         # 256 + 255 < 512: no frame yet
    out = pp.process(np.zeros(1, np.int16))                          # exactly 512 padded samples -> 1 frame
    assert out.shape[0] == 1
    assert np.allclose(out, np.log(np.float32(2.0 ** -24)))         # silence -> log(zero guard)
    full = O.Preproc(model=model2).process(np.full(4000, -32768, np.int16))   # full-scale negative DC
    assert np.isfinite(full).all()


def test_model_math_matches_reference_golden(built, model2):
    g = np.load(os.path.join(GOLD, "model_ref_L2.npz"))
    sub = model2.subsampling(g["chunk"])
    assert sub.shape == g["sub"].shape == (4, 1024)                   # T + 2 frames for R = 1 (M = 25)
    assert np.abs(sub - g["sub"]).max() <= 1e-4 * np.abs(g["sub"]).max()
    # first streaming chunk (cache empty => fully masked) == the reference's non-cached layers after drop-2
    s = O.Stream(model2, 1, trace=True)
    assert s.push_mel(g["chunk"][9:]) == 1
    assert np.abs(s.last_sub() - g["sub"][2:]).max() <= 1e-4 * np.abs(g["sub"]).max()
    for l, key in enumerate(("layer0", "layer1")):
        assert np.abs(s.last_layer(l) - g[key]).max() <= 1e-4 * np.abs(g[key]).max(), key
    assert np.abs(s.trace_logits(0) - g["logits0"]).max() <= 1e-4 * np.abs(g["logits0"]).max()
    assert np.array_equal(s.tokens(), g["tokens"])                    # greedy: exact token match (test_compute.cpp:2808-2820)


@pytest.mark.skipif(not O.ref_available(), reason="oracle/_ref/libnemo_ref.so not built (needs a reference checkout, NSB_REFERENCE_DIR)")
def test_against_compiled_reference_all_latency_modes(built, model2):
    fb, win = synth.mel_filterbank(), synth.gen_tensor("w", (400,), ("window", 0), 1234, 0, 0)
    pcm = synth.synth_pcm(5, 1.5)
    mel_o = O.Preproc(model=model2).process(pcm)
    mel_r = O.RefPreproc(fb, win).process(pcm)
    assert np.array_equal(mel_o.view(np.uint32), mel_r.view(np.uint32))
    rw = O.RefWeights(synth.cached_model("nemo", 2, R=0))
    for R in (0, 1, 6, 13):
        T, M = 1 + R, 9 + 8 * (1 + R)
        chunk = np.concatenate([np.zeros((9, 128), np.float32), mel_o[:8 * T]])
        sub_r = rw.subsampling(chunk)
        assert sub_r.shape[0] == T + 2                                # t3 = T + 2 (SURVEY appendix B)
        s = O.Stream(model2, R, trace=True)
        assert s.push_mel(mel_o[:8 * T]) == 1
        x = sub_r[2:]
        for l in range(2):
            x = rw.layer(l, x)
            assert np.abs(s.last_layer(l) - x).max() <= 1e-4 * np.abs(x).max(), (R, l)
        assert np.array_equal(s.tokens(), rw.greedy(x)), R


def _cached_stream_from_reference_modules(model2, rw, R, secs):
    """Free-running streaming encoder built ONLY from the reference's compiled code: ConvSubsampling::forward on [9 carried mel
    frames | chunk] minus the 2 pre-encode frames, then per layer ref_cached_layer_step (the modules ConformerLayer::forward calls,
    run on [history | chunk] windows), then GreedyDecoder::decode over all frames (= chunked greedy with carried state)."""
    T = 1 + R
    mel = O.Preproc(model=model2).process(synth.synth_pcm(11, secs))
    s = O.Stream(model2, R, trace=True)
    att = [np.zeros((0, 1024), np.float32) for _ in range(2)]
    conv = [np.zeros((0, 1024), np.float32) for _ in range(2)]
    carry, encs, worst = np.zeros((9, 128), np.float32), [], 0.0
    n_chunks = len(mel) // (8 * T)
    for c in range(n_chunks):
        new = mel[8 * T * c:8 * T * (c + 1)]
        assert s.push_mel(new) == 1
        chunk = np.concatenate([carry, new]); carry = chunk[-9:]
        x = rw.subsampling(chunk)[2:]
        worst = max(worst, float(np.abs(x - s.last_sub()).max() / np.abs(x).max()))
        for l in range(2):
            x, att[l], conv[l] = rw.cached_layer_step(l, x, att[l], conv[l])
            worst = max(worst, float(np.abs(x - s.last_layer(l)).max() / np.abs(x).max()))
        encs.append(x)
    return n_chunks, worst, rw.greedy(np.concatenate(encs)), s.tokens()


@pytest.mark.skipif(not O.ref_available(), reason="oracle/_ref/libnemo_ref.so not built (needs a reference checkout, NSB_REFERENCE_DIR)")
def test_cached_streaming_steps_match_reference_modules_past_the_cache_roll(built, model2):
    """Pins the CACHED step (K/V cache + mask + rel-shift over K = 70 + T keys, conv cache, cache roll once more than 70 frames
    went by, decoder state carried across chunks) -- the part no runnable reference test covers -- against the reference's own
    compiled modules in every latency mode: the caching is restated as windows over the non-cached modules
    (oracle/ref_shim.cpp:ref_cached_layer_step), everything else is the reference's code. Encoder tensors per chunk and layer
    <= 1e-4 relative (measured 2e-6), greedy tokens identical."""
    from concurrent.futures import ThreadPoolExecutor
    rw = O.RefWeights(synth.cached_model("nemo", 2, R=0))
    cases = [(0, 6.0), (1, 6.6), (6, 7.5), (13, 9.0)]                 # 74 / 82 / 91 / 112 encoder frames: all roll the 70-row cache
    with ThreadPoolExecutor(4) as ex:                                  # the naive reference loops dominate; ctypes drops the GIL
        results = list(ex.map(lambda a: _cached_stream_from_reference_modules(model2, rw, *a), cases))
    for (R, _), (n_chunks, worst, ref_tokens, tokens) in zip(cases, results):
        assert n_chunks * (1 + R) > 70 + (1 + R), R
        assert worst <= 1e-4, (R, worst)
        assert len(tokens) > 0 and np.array_equal(ref_tokens, tokens), R


@pytest.mark.parametrize("R,secs", [(0, 6.0), (1, 6.6), (6, 7.5), (13, 9.0)])
def test_cached_streaming_matches_reference_golden(built, model2, R, secs):
    """The committed fixture of the test above (tests/golden/cached_ref_L2.npz, tools/make_golden.py section 3): holds where
    no reference checkout is available. All tokens of the stream + the encoder output of the last chunk (cache rolled)."""
    g = np.load(os.path.join(GOLD, "cached_ref_L2.npz"))
    s = O.Stream(model2, R, trace=True)
    s.push(synth.synth_pcm(11, secs))
    assert s.chunks == int(g[f"chunks_R{R}"])
    want = g[f"enc_last_R{R}"]
    assert np.abs(s.last_layer(1) - want).max() <= 1e-4 * np.abs(want).max()
    assert np.array_equal(s.tokens(), g[f"tokens_R{R}"])


@pytest.mark.skipif(not O.ref_available(), reason="oracle/_ref/libnemo_ref.so not built (needs a reference checkout, NSB_REFERENCE_DIR)")
def test_batch_path_matches_compiled_reference(built, model2):
    """SURVEY 8f.1, oracle side only (no CUDA batch path yet): the non-streaming nemo_encode path -- whole-utterance subsampling
    with no carried / dropped frames, non-cached layers, greedy from a fresh decoder state -- against the reference's compiled
    ConvSubsampling / ConformerLayer / GreedyDecoder."""
    pcm = synth.synth_pcm(21, 3.0)
    mel = O.Preproc(model=model2).process(pcm)
    enc, toks, frames = model2.transcribe_full(mel)
    rw = O.RefWeights(synth.cached_model("nemo", 2, R=0))
    x = rw.subsampling(mel)
    assert x.shape[0] == enc.shape[0] == ((len(mel) // 2 + 1) // 2 + 1) // 2 + 1            # three stride-2 convs with (2, 1) padding
    for l in range(2):
        x = rw.layer(l, x)
    assert np.abs(enc - x).max() <= 1e-4 * np.abs(x).max()
    assert len(toks) > 0 and np.array_equal(toks, rw.greedy(x))
    assert np.all(np.diff(frames) >= 0) and frames.max() < enc.shape[0] and np.bincount(frames).max() <= 10


def test_batch_path_matches_reference_golden(built, model2):
    g = np.load(os.path.join(GOLD, "batch_ref_L2.npz"))              # tools/make_golden.py section 4
    mel = O.Preproc(model=model2).process(synth.synth_pcm(21, 3.0))
    assert len(mel) == int(g["n_mel"])
    enc, toks, _ = model2.transcribe_full(mel)
    assert np.abs(enc[::4] - g["enc_every4"]).max() <= 1e-4 * np.abs(g["enc_every4"]).max()
    assert np.array_equal(toks, g["tokens"])


def test_chunk_arithmetic_matches_reference_worked_example(built, model2):
    # SURVEY 8(a) row D (from nemo-stream.h:65-100, nemo-stream.cpp:1094-1127): 10 s, R = 13 -> 999 mel frames, 8 chunks
    pcm = synth.synth_pcm(1, 10.0)
    assert len(pcm) == 160000
    s = O.Stream(model2, 13)
    s.push(pcm)
    assert s.chunks == 8
    for R, n_chunks_5s in ((0, None), (1, None), (6, None)):
        T = 1 + R
        n = 80000
        frames = (256 + n - 512 + 160) // 160
        expect = (9 + frames - (9 + 8 * T)) // (8 * T) + 1
        st = O.Stream(model2, R)
        st.push(pcm[:n])
        assert st.chunks == expect, (R, st.chunks, expect)


def test_streaming_is_push_granularity_independent(built, model2):
    pcm = synth.synth_pcm(9, 2.0)
    a = O.Stream(model2, 1); a.push(pcm)
    b = O.Stream(model2, 1)
    for i in range(0, len(pcm), 4000):                                 # CLI read size for R = 1 (160 * 25)
        b.push(pcm[i:i + 4000])
    c = O.Stream(model2, 1)
    for i in range(0, len(pcm), 333):
        c.push(pcm[i:i + 333])
    assert a.chunks == b.chunks == c.chunks
    assert np.array_equal(a.tokens(), b.tokens()) and np.array_equal(a.tokens(), c.tokens())
    assert len(a.tokens()) > 0


def test_cache_carry_over_self_consistency(built, model2):
    """Not pinned by any reference test ("parity unpinned" boundary): check the properties the disabled reference
    tests were after (tests/test_streaming.cpp:463-511): the conv cache holds the last 8 GLU rows and the K/V cache the
    last 70 rows in order; cache_valid_len saturates at 70."""
    s = O.Stream(model2, 6, trace=True)
    pcm = synth.synth_pcm(2, 7.5)
    s.push(pcm)
    assert s.chunks >= 11
    import ctypes
    assert O.lib().orc_stream_cache_valid(s.h) == 70
    k = s.cache(0, 0)
    assert np.abs(k).max() > 0 and np.isfinite(k).all()
    # with R = 6 the last 7 cache rows are the K rows of the last chunk; re-running the last chunk's layer input through
    # linear_k must reproduce them: use the trace of a second stream stopped one chunk earlier
    s2 = O.Stream(model2, 6, trace=True)
    need = 160 * (8 * 7 * (s.chunks - 1) - 1) + 256
    s2.push(pcm[:need])
    assert s2.chunks == s.chunks - 1
    k_prev = s2.cache(0, 0)
    assert np.array_equal(k[:63], k_prev[7:])                           # roll by T = 7 rows (nemo-stream.cpp:477-484)


def test_q8_0_activation_quantisation_matches_gguf_package(built):
    """ggml semantics for Q8_0 weights (SURVEY 8c): activations are quantised per 32 with d = amax/127 (fp16),
    q = round(x/d); block dots are integer; pinned against the gguf python package (bit-exact with ggml-quants.c)."""
    import gguf
    from gguf import quants
    path = synth.cached_model("q8_0", 2, R=0)
    m = O.Model(path, O.MM_REF)
    name = "encoder.layers.0.self_attn.linear_q.weight"
    rng = np.random.default_rng(3)
    x = rng.standard_normal((3, 1024)).astype(np.float32)
    y = m.matmul(name, x)
    r = gguf.GGUFReader(path)
    t = [t for t in r.tensors if t.name == name][0]
    w = quants.dequantize(t.data, t.tensor_type).astype(np.float64)                     # d_w * q_w
    xq = quants.dequantize(quants.quantize(x, gguf.GGMLQuantizationType.Q8_0), gguf.GGMLQuantizationType.Q8_0).astype(np.float64)
    ref = xq @ w.T
    assert np.abs(y - ref).max() <= 2e-6 * np.abs(ref).max()


def test_q4_0_weights_match_gguf_package(built):
    """Q4_0 files (the converter's other quantised type, convert_to_gguf.py:132-179): the synthetic writer's blocks dequantise
    to the same values as the gguf package's (nibble order, d = amax / 7), and the oracle's ggml-semantics matmul
    (Q8_0-quantised activations x Q4_0 weights, integer block dots) agrees with that arithmetic done in numpy."""
    import gguf
    from gguf import quants
    path = synth.cached_model("q4_0", 2, R=0)
    r = gguf.GGUFReader(path)
    name = "encoder.layers.0.self_attn.linear_q.weight"
    t = [t for t in r.tensors if t.name == name][0]
    assert t.tensor_type.name == "Q4_0"
    w = quants.dequantize(t.data, t.tensor_type).astype(np.float64)                     # d_w * (q_w - 8)
    wf = [t for t in gguf.GGUFReader(synth.cached_model("f32", 2, R=0)).tensors if t.name == name][0].data.astype(np.float64)
    assert np.abs(w - wf.reshape(w.shape)).max() <= np.abs(wf).max() / 7.0 * 0.51 + 1e-6  # within half a quantisation step (+ fp16 d)
    m = O.Model(path, O.MM_REF)
    rng = np.random.default_rng(4)
    x = rng.standard_normal((3, 1024)).astype(np.float32)
    y = m.matmul(name, x)
    xq = quants.dequantize(quants.quantize(x, gguf.GGMLQuantizationType.Q8_0), gguf.GGMLQuantizationType.Q8_0).astype(np.float64)
    ref = xq @ w.T
    assert np.abs(y - ref).max() <= 2e-6 * np.abs(ref).max()
    # engine-mirror arithmetic (weights expanded to fp16 once, fp16 activations): close to the exact product of the dequantised values
    y2 = O.Model(path, O.MM_Q8FAST).matmul(name, x)
    assert np.abs(y2 - x.astype(np.float64) @ w.T).max() <= 3e-3 * np.abs(ref).max()


def test_synthetic_gguf_layout_is_readable_by_gguf_package(built):
    import gguf
    for kind in ("f32", "f16", "q8_0", "q4_0"):
        r = gguf.GGUFReader(synth.cached_model(kind, 2, R=0))
        assert len(r.tensors) == 12 + 2 * 26 + 9 + 6 + 2
        names = {t.name: t for t in r.tensors}
        dw = names["encoder.layers.0.conv.depthwise_conv.weight"]
        assert list(dw.shape) == [1024, 9] and dw.tensor_type.name == "F32"          # tap-major, never quantised
        lin = names["encoder.layers.1.feed_forward1.linear1.weight"]
        assert lin.tensor_type.name == {"f32": "F32", "f16": "F16", "q8_0": "Q8_0", "q4_0": "Q4_0"}[kind]
        assert names["joint.enc.weight"].tensor_type.name == "F32"
        assert names["encoder.pre_encode.out.weight"].tensor_type.name == "F32"
        keys = list(r.fields.keys())
        assert keys.index("tokenizer.vocab") < keys.index("nemo.n_mels")


def test_detokeniser(built, model2):
    # tokens_to_text (src/nemo-ggml.cpp:1432-1458): U+2581 prefix -> ' ' + rest; out-of-range ids skipped
    vocab = bytes((O.lib().orc_model_vocab(model2.h) and __import__("ctypes").string_at(O.lib().orc_model_vocab(model2.h), 1025 * 8)))
    pieces = [vocab[i * 8:(i + 1) * 8].split(b"\0")[0].decode() for i in range(1025)]
    ids = [i for i in range(50)] + [1024, 5000, -1]
    expect = "".join((" " + p[1:]) if p.startswith("▁") else p for p in (pieces[i] for i in range(50)))
    assert model2.detok(ids) == expect


@pytest.mark.skipif(not O.reference_file("scripts/compare_tensors.py"), reason="no reference checkout (NSB_REFERENCE_DIR)")
def test_encoder_dump_is_readable_by_the_reference_compare_script(built, model2, tmp_path):
    """tools/dump_encoder_out.py writes per-chunk encoder output in the reference's own dump format (nemo-stream.cpp:886-958); the
    reference's scripts/compare_tensors.py must load it (its loader reads the first chunk) and report it identical to itself."""
    import importlib.util
    import subprocess
    import sys
    pcm = synth.synth_pcm(4, 1.2)
    f = tmp_path / "a.pcm"; pcm.tofile(f)
    out = tmp_path / "enc.bin"
    tool = os.path.join(os.path.dirname(GOLD), "..", "tools", "dump_encoder_out.py")
    subprocess.check_call([sys.executable, tool, "--impl", "oracle", synth.cached_model("f32", 2, R=0), str(f), "6", str(out)])
    spec = importlib.util.spec_from_file_location("ref_compare_tensors", O.reference_file("scripts/compare_tensors.py"))
    ref = importlib.util.module_from_spec(spec); spec.loader.exec_module(ref)
    t = ref.load_tensor(str(out))
    s = O.Stream(model2, 6, trace=True); s.push(pcm)
    assert s.chunks == 2 and t.shape == (7, 1024)
    assert np.array_equal(t, s.trace_enc(0))
    assert os.path.getsize(out) == 32 + s.chunks * 7 * 1024 * 4
