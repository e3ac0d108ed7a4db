"""CPU tests of the boundary: the C-ABI library loads and exports every symbol include/nsb200.h declares, the
GGUF probe works without a GPU, engine creation fails loudly (no CPU fallback), and the reference's own CLI source
compiles UNMODIFIED against the drop-in headers (include/nemo-ggml.h, include/nemo-stream.h)."""
import os
import re
import subprocess

import numpy as np
import pytest

import oracle as O
import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol(built):
    import nsb200
    hdr = open(os.path.join(ROOT, "include", "nsb200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    declared = sorted(set(re.findall(r"\b(nsb_[a-z0-9_]+)\s*\(", hdr)))
    assert len(declared) >= 25
    out = subprocess.check_output(["nm", "-D", "--defined-only", nsb200.LIB_PATH], text=True)
    exported = set(re.findall(r" T (nsb_[a-z0-9_]+)", out))
    missing = [d for d in declared if d not in exported]
    assert not missing, missing
    L = nsb200.lib()
    assert all(hasattr(L, n) for n in nsb200.EXPORTS)
    assert sorted(nsb200.EXPORTS) == [d for d in declared], set(declared) ^ set(nsb200.EXPORTS)


def test_library_is_tensor_core_native(built):
    """SASS evidence that the shipped .so holds tcgen05 / TMEM / TMA code (B200_PROFILING.md mnemonics)."""
    import nsb200
    sass = subprocess.run(["cuobjdump", "-sass", nsb200.LIB_PATH], capture_output=True, text=True).stdout
    if not sass:
        pytest.skip("cuobjdump unavailable")
    for mnemonic in ("UTCHMMA", "UTMALDG", "LDTM"):
        assert mnemonic in sass, mnemonic
    assert "sm_100a" in sass


def test_gguf_probe_and_errors(built, tmp_path):
    import nsb200
    info = nsb200.probe(synth.cached_model("q8_0", 2, R=0))
    assert (info.n_layers, info.d_model, info.vocab_size, info.n_tensors, info.weight_type) == (2, 1024, 1025, 81, 8)
    assert nsb200.probe(synth.cached_model("f32", 2, R=0)).weight_type == 0
    assert nsb200.probe(synth.cached_model("q4_0", 2, R=0)).weight_type == 2          # Q4_0 blocks (18 bytes per 32 weights) are sized and located
    with pytest.raises(nsb200.NsbError, match="cannot open"):
        nsb200.probe(str(tmp_path / "missing.gguf"))
    bad = tmp_path / "bad.gguf"
    bad.write_bytes(b"NOPE" + b"\0" * 64)
    with pytest.raises(nsb200.NsbError, match="bad magic"):
        nsb200.probe(str(bad))
    trunc = tmp_path / "trunc.gguf"
    trunc.write_bytes(open(synth.cached_model("f32", 2, R=0), "rb").read(3000))
    with pytest.raises(nsb200.NsbError):
        nsb200.probe(str(trunc))
    # complete header, tensor data cut short (an interrupted download): refused at open, naming the first tensor that does not fit
    full = open(synth.cached_model("f32", 2, R=0), "rb").read()
    cut = tmp_path / "cut.gguf"
    cut.write_bytes(full[:len(full) - 4096])
    with pytest.raises(nsb200.NsbError, match="file truncated: tensor '"):
        nsb200.probe(str(cut))


def test_no_cpu_fallback(built):
    """Without a usable sm_100 device the engine must refuse to exist (never a silent CPU path)."""
    import torch
    import nsb200
    if torch.cuda.is_available():
        pytest.skip("GPU present: covered by the -m gpu suite")
    with pytest.raises(nsb200.NsbError, match="no CUDA device"):
        nsb200.Engine(synth.cached_model("f32", 2, R=0))


def test_product_sources_do_not_touch_the_oracle():
    pkg = os.path.join(ROOT, "nemotron-speech.cpp_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".cu", ".cuh", ".cpp", ".h", ".py", "Makefile")):
                txt = open(os.path.join(dirpath, f), errors="ignore").read()
                assert "oracle" not in txt.lower().replace("# oracle", ""), os.path.join(dirpath, f)
    for f in ("include/nsb200.h", "include/nemo-ggml.h", "include/nemo-stream.h", "include/preprocessor.h", "nsb200.py"):
        assert "liboracle" not in open(os.path.join(ROOT, f)).read()


@pytest.mark.skipif(not O.reference_file("src/transcribe_stream.cpp"), reason="no reference checkout (NSB_REFERENCE_DIR)")
def test_reference_cli_compiles_unmodified_against_dropin_headers(built, tmp_path):
    exe = tmp_path / "nemotron-asr"
    pkg = os.path.join(ROOT, "nemotron-speech.cpp_b200")
    # a quoted #include looks next to the source file first, so build a byte-identical copy outside the reference tree
    src = tmp_path / "transcribe_stream.cpp"
    src.write_bytes(open(O.reference_file("src/transcribe_stream.cpp"), "rb").read())
    cmd = ["/usr/bin/g++", "-std=c++17", "-O2", "-I", os.path.join(ROOT, "include"), str(src),
           "-L", pkg, "-lnsb200", f"-Wl,-rpath,{pkg}", "-o", str(exe)]
    subprocess.check_call(cmd)
    r = subprocess.run([str(exe)], capture_output=True, text=True)            # argc < 3 -> usage, exit 1 (transcribe_stream.cpp:53-56)
    assert r.returncode == 1 and "Usage:" in r.stderr
    r = subprocess.run([str(exe), str(tmp_path / "none.gguf"), "-"], capture_output=True, text=True, input="")
    assert r.returncode == 1 and "Failed to load model" in r.stderr          # :102-105


@pytest.mark.skipif(not O.reference_file("src/transcribe.cpp"), reason="no reference checkout (NSB_REFERENCE_DIR)")
def test_reference_batch_cli_compiles_unmodified_against_dropin_headers(built, tmp_path):
    """src/transcribe.cpp (the non-streaming CLI) against include/: nemo_transcribe_audio exists in the shim (its CUDA side is
    experimental this round); usage and load-failure behaviour are the reference's (transcribe.cpp:31-34,52-56)."""
    exe = tmp_path / "nemotron-asr-batch"
    pkg = os.path.join(ROOT, "nemotron-speech.cpp_b200")
    # it includes "../src/nemo-ggml.h": lay the tree out as a maintainer who adopted the drop-in would (INTEGRATION.md section 2:
    # src/nemo-ggml.h replaced by include/nemo-ggml.h), the CLI source byte-identical
    import shutil
    (tmp_path / "src").mkdir()
    for h in os.listdir(os.path.join(ROOT, "include")):
        shutil.copy(os.path.join(ROOT, "include", h), tmp_path / "src" / h)
    src = tmp_path / "src" / "transcribe.cpp"
    src.write_bytes(open(O.reference_file("src/transcribe.cpp"), "rb").read())
    subprocess.check_call(["/usr/bin/g++", "-std=c++17", "-O2", "-I", os.path.join(ROOT, "include"), str(src),
                           "-L", pkg, "-lnsb200", f"-Wl,-rpath,{pkg}", "-o", str(exe)])
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    assert r.returncode == 1
    r = subprocess.run([str(exe), str(tmp_path / "none.gguf"), str(tmp_path / "a.pcm")], capture_output=True, text=True)
    assert r.returncode == 1 and "Failed to load model" in r.stderr


HEADER_PROBE = r"""
#include "nemo-stream.h"
#include <cstdio>
int main() {
    const nemo_cache_config modes[] = {nemo_cache_config::default_config(), nemo_cache_config::pure_causal(), nemo_cache_config::ultra_low_latency(),
                                       nemo_cache_config::low_latency(), nemo_cache_config::balanced(),
                                       nemo_cache_config::with_latency(nemo_latency_mode::LOW)};
    for (const nemo_cache_config& c : modes)
        printf("cfg R=%d L=%d chunk_mel=%zu shift_mel=%zu samples=%d latency_ms=%d valid_out=%d k=%d cc=%d drop=%d pre=%d blank=%d vocab=%d hop=%d sr=%d\n",
               (int)c.att_right_context, (int)c.att_left_context, (size_t)c.get_chunk_mel_frames(), (size_t)c.get_shift_mel_frames(),
               (int)c.get_chunk_samples(), (int)c.get_latency_ms(), (int)c.get_valid_out_len(), (int)c.conv_kernel_size, (int)c.conv_cache_size,
               (int)c.drop_extra_pre_encoded, (int)c.pre_encode_cache_size, (int)c.blank_token, (int)c.vocab_size, (int)c.hop_length, (int)c.sample_rate);
    printf("modes %d %d %d %d\n", (int)nemo_latency_mode::PURE_CAUSAL, (int)nemo_latency_mode::ULTRA_LOW, (int)nemo_latency_mode::LOW, (int)nemo_latency_mode::DEFAULT);
    nemo_decoder_state d;
    printf("dec fresh init=%d prev=%d\n", (int)d.is_initialized(), d.prev_token);
    d.init(2, 640); d.prev_token = 7; d.h[5] = 1.5f; d.c[700] = -2.f; d.frame_offset = 9;
    printf("dec set init=%d h=%zu c=%zu hl1=%ld\n", (int)d.is_initialized(), d.h.size(), d.c.size(), (long)(d.h_layer(1) - d.h.data()));
    d.reset(1024);
    printf("dec reset prev=%d h5=%g c700=%g off=%ld init=%d\n", d.prev_token, d.h[5], d.c[700], (long)d.frame_offset, (int)d.is_initialized());
    d.reset();
    printf("dec reset0 prev=%d init=%d\n", d.prev_token, (int)d.is_initialized());
    timed_token t(42, 25);
    printf("tok %d %ld %.4f %.4f\n", t.token_id, (long)t.frame_idx, t.to_seconds(), t.to_seconds(640, 8000));
    nemo_hparams hp;
    printf("hp %d %d %d %d %d %d %d %d\n", hp.n_mels, hp.d_model, hp.n_heads, hp.d_head, hp.d_ff, hp.n_layers, hp.vocab_size, hp.joint_dim);
    printf("backend %d %d %d %d\n", (int)NEMO_BACKEND_CPU, (int)NEMO_BACKEND_CUDA, (int)NEMO_BACKEND_METAL, (int)NEMO_BACKEND_AUTO);
    return 0;
}
"""

GGML_STUB = """#pragma once
#include <cstddef>
#include <cstdint>
struct ggml_tensor; struct ggml_context; struct ggml_cgraph; struct gguf_context;
typedef struct ggml_backend* ggml_backend_t; typedef struct ggml_backend_buffer* ggml_backend_buffer_t; typedef struct ggml_gallocr* ggml_gallocr_t;
"""


def test_dropin_headers_agree_with_the_reference_headers(tmp_path):
    """Differential test of the host-side logic that lives in the headers (what the reference's tests/test_streaming.cpp unit
    tests poke: chunk / shift / latency arithmetic of every latency mode and factory, nemo_decoder_state init / reset,
    timed_token::to_seconds, hparams defaults, enum values): the probe compiled against include/ must print what it printed
    compiled against the REFERENCE's own src/nemo-stream.h + src/nemo-ggml.h (ggml's headers replaced by empty forward-declaration
    stubs; header-only, nothing of the reference is linked). That output is committed (tests/golden/header_probe_ref.txt); with a
    reference checkout the probe is also compiled against its headers again."""
    stub = tmp_path / "stub"; stub.mkdir()
    (stub / "ggml.h").write_text(GGML_STUB)
    for h in ("ggml-cpu.h", "ggml-alloc.h", "ggml-backend.h", "gguf.h"):
        (stub / h).write_text("#pragma once\n")
    src = tmp_path / "probe.cpp"
    src.write_text(HEADER_PROBE)
    with open(os.path.join(ROOT, "tests", "golden", "header_probe_ref.txt")) as f:
        outs = [f.read()]
    builds = [("ours", [os.path.join(ROOT, "include")])]
    if O.reference_file("src/nemo-stream.h"):
        builds.append(("ref", [str(stub), O.reference_file("src")]))
    for name, incs in builds:
        exe = tmp_path / f"probe_{name}"
        cmd = ["/usr/bin/g++", "-std=c++17", "-O1"] + [f"-I{i}" for i in incs] + [str(src), "-o", str(exe)]
        subprocess.check_call(cmd)
        outs.append(subprocess.check_output([str(exe)], text=True))
    for out in outs[1:]:
        assert out == outs[0], "\n--- reference headers\n" + outs[0] + "--- this build\n" + out
    assert "chunk_mel=121" in outs[1] and "samples=19360" in outs[1] and "latency_ms=1210" in outs[1]      # R = 13 (SURVEY appendix B)


DETOK_PROBE = r"""
#include "nemo-ggml.h"
#include <cstdio>
#include <cstring>
int main() {
    const char* pieces[] = {"\xe2\x96\x81he", "llo", "\xe2\x96\x81wor", "ld", "abcdefgh", "\xe2\x96\x81", ""};
    std::vector<char8> vocab(7);
    for (int i = 0; i < 7; ++i) { memset(vocab[i].data, 0, 8); memcpy(vocab[i].data, pieces[i], strlen(pieces[i]) > 8 ? 8 : strlen(pieces[i])); }
    std::vector<timed_token> t = {{0, 0}, {1, 1}, {2, 12}, {3, 13}, {-1, 14}, {99, 15}, {4, 16}, {5, 20}, {6, 21}};
    printf("[%s]\n[%s]\n", tokens_to_text(t, vocab, false).c_str(), tokens_to_text(t, vocab, true).c_str());
    return 0;
}
"""


def test_tokens_to_text_of_the_shim(built, tmp_path):
    """tokens_to_text (src/nemo-ggml.cpp:1432-1458) as exported by the drop-in library: U+2581 -> space, out-of-range ids skipped,
    "{seconds}" after the space in timestamp mode (frame * 1280 / 16000), and an 8-byte piece without a NUL does not run on into
    its neighbour (the reference reads it as a C string)."""
    pkg = os.path.join(ROOT, "nemotron-speech.cpp_b200")
    src = tmp_path / "detok.cpp"; src.write_text(DETOK_PROBE)
    exe = tmp_path / "detok"
    subprocess.check_call(["/usr/bin/g++", "-std=c++17", "-O1", "-I", os.path.join(ROOT, "include"), str(src), "-L", pkg, "-lnsb200",
                           f"-Wl,-rpath,{pkg}", "-o", str(exe)])
    out = subprocess.check_output([str(exe)], text=True).splitlines()
    assert out[0] == "[ hello worldabcdefgh ]"
    assert out[1] == "[ {0.00}hello {0.96}worldabcdefgh {1.60}]"


HOST_STREAM_PROBE = r"""
#include "host_stream.h"
#include <cstdio>
#include <cstdlib>
#include <random>
using namespace nsb;
// usage: probe T n_samples seed  -> pushes a seeded PCM stream in ragged pieces, stages every due chunk's row, checks it against
// the definition (raw[1280 T c - 257 + k], zeros before the stream start) and prints the number of chunks
int main(int argc, char** argv) {
    const int T = atoi(argv[1]); const long long n = atoll(argv[2]); std::mt19937 rng(atoi(argv[3]));
    std::vector<int16_t> pcm((size_t)n);
    for (auto& v : pcm) v = (int16_t)(rng() % 65536 - 32768);
    HostStream h; h.open = true;
    const int rl = hs_row_len(T);
    if (rl != 1280 * T + 353) { printf("FAIL row_len\n"); return 1; }
    std::vector<int16_t> row((size_t)rl);
    long long pos = 0; int chunks = 0; size_t max_buf = 0;
    while (pos < n) {
        const long long k = std::min<long long>(n - pos, 1 + rng() % 5000);
        hs_push(h, pcm.data() + pos, (int)k); pos += k;
        while (hs_ready(h, T)) {
            hs_stage_row(h, T, rl, row.data());
            const long long start = 1280LL * T * chunks - 257;
            for (int i = 0; i < rl; ++i) {
                const long long idx = start + i;
                const int16_t want = idx < 0 ? 0 : pcm[(size_t)idx];
                if (idx >= pos) { printf("FAIL chunk %d reads sample %lld beyond the %lld pushed\n", chunks, idx, pos); return 1; }
                if (row[i] != want) { printf("FAIL chunk %d sample %d\n", chunks, i); return 1; }
            }
            hs_launched(h, T); ++chunks;
            max_buf = std::max(max_buf, h.buf.size());
        }
    }
    // the gate is tight: one more chunk needs exactly 160 (8T (c+1) - 1) + 256 samples
    if (n >= 160LL * (8LL * T * (chunks + 1) - 1) + 256) { printf("FAIL gate\n"); return 1; }
    printf("%d %zu\n", chunks, max_buf);
    return 0;
}
"""


def test_host_stream_bookkeeping_against_the_oracle(built, tmp_path):
    """csrc/host_stream.h is the engine's host-side chunk gate + PCM staging (pure C++): ragged pushes, every staged row checked
    against its definition, chunk counts == the oracle's streaming driver (nemo-stream.cpp:1094-1127) for the same lengths, and the
    retained buffer stays bounded (one row + one push)."""
    import oracle as O
    src = tmp_path / "hs.cpp"; src.write_text(HOST_STREAM_PROBE)
    exe = tmp_path / "hs"
    subprocess.check_call(["/usr/bin/g++", "-std=c++17", "-O1", "-I", os.path.join(ROOT, "nemotron-speech.cpp_b200", "csrc"), str(src), "-o", str(exe)])
    om = O.Model(synth.cached_model("f32", 2, R=0))
    rng = np.random.default_rng(5)
    for R in (0, 1, 6, 13):
        T = R + 1
        for n in [95, 1280 * T + 95, 1280 * T + 96, 1280 * T + 97, int(rng.integers(20000, 60000)), 160 * (8 * T * 3 - 1) + 256]:
            out = subprocess.check_output([str(exe), str(T), str(n), str(R * 7 + 1)], text=True).split()
            assert out[0] != "FAIL", (R, n, out)
            chunks, max_buf = int(out[0]), int(out[1])
            assert max_buf <= (1280 * T + 353) + 5000 + 1280 * T
            if n <= 30000:                                               # the oracle runs the model: keep its share small
                st = O.Stream(om, R); st.push(np.zeros(n, np.int16))
                assert st.chunks == chunks, (R, n, st.chunks, chunks)
            assert chunks == max(0, (n - 96) // (1280 * T))


@pytest.mark.parametrize("kind", ["f16", "q8_0", "q4_0"])
def test_product_loader_dequantisation_matches_gguf_package(built, kind):
    """The engine's own GGUF reader (csrc/gguf_loader.cpp through nsb_gguf_read_tensor, no GPU): every tensor of a synthetic file
    of each weight type, bit for bit against the gguf package's reader + dequantiser (documented bit-exact with ggml-quants.c)."""
    import gguf
    import nsb200
    path = synth.cached_model(kind, 2, R=0)
    rd = gguf.GGUFReader(path)
    seen = set()
    for t in rd.tensors:
        want = gguf.quants.dequantize(np.asarray(t.data), t.tensor_type).astype(np.float32).reshape(-1)
        got, ty = nsb200.read_tensor(path, t.name)
        assert ty == int(t.tensor_type) and got.shape == want.shape, t.name
        assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), t.name
        seen.add(ty)
    assert {"f16": 1, "q8_0": 8, "q4_0": 2}[kind] in seen and 0 in seen
    with pytest.raises(nsb200.NsbError, match="missing tensor"):
        nsb200.read_tensor(path, "encoder.layers.99.nope")


def test_c_abi_header_is_plain_c_and_the_example_runs_on_the_test_double(tmp_path):
    """include/nsb200.h must be consumable from plain C (the boundary other hosts bind: cgo, JNI, N-API ... all speak C):
    examples/minimal.c compiles as strict C99 (-pedantic -Werror) and, linked against the test double of the library
    (tests/mock_nsb200.cpp), runs the push / step / pop / detokenise sequence."""
    obj = tmp_path / "minimal.o"
    subprocess.check_call(["gcc", "-std=c99", "-pedantic", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"), "-c",
                           os.path.join(ROOT, "examples", "minimal.c"), "-o", str(obj)])
    exe = tmp_path / "minimal"
    subprocess.check_call(["/usr/bin/g++", "-std=c++17", "-O1", "-I", os.path.join(ROOT, "include"), "-I",
                           os.path.join(ROOT, "nemotron-speech.cpp_b200", "csrc"), str(obj), os.path.join(ROOT, "tests", "mock_nsb200.cpp"), "-o", str(exe)])
    f = tmp_path / "a.pcm"
    np.zeros(16000 * 3, np.int16).tofile(f)
    r = subprocess.run([str(exe), str(tmp_path / "model.gguf"), str(f), "1"], capture_output=True, text=True)
    chunks = (48000 - 96) // 2560
    assert r.returncode == 0 and r.stdout == "".join(f"<{c}>" for c in range(chunks)) + "\n", (r.stdout, r.stderr)
    assert f"{chunks} chunks, {chunks} tokens" in r.stderr
