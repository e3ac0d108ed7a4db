"""nemotron-asr-serve (csrc/serve_main.cpp): the multi-stream / multi-GPU host program over the C ABI.
CPU: argument handling and the reference CLI's failure behaviour (exit code 1 + "Failed to load model" / "Failed to open audio
file", transcribe_stream.cpp:102-105,131-137), no CPU fallback. GPU: transcripts of ragged streams run in waves through the
batched engine == the oracle's per-stream transcripts; --flush == the oracle on zero-padded audio; --realtime == throughput mode."""
import os
import subprocess

import numpy as np
import pytest

import oracle as O
import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "nemotron-speech.cpp_b200", "nemotron-asr-serve")


@pytest.fixture(scope="module")
def exe(built):
    if not os.path.exists(EXE):
        subprocess.check_call(["make", "-C", os.path.dirname(EXE), "nemotron-asr-serve"], stdout=subprocess.DEVNULL)
    return EXE


def run(exe, *args, timeout=300):
    return subprocess.run([exe, *map(str, args)], capture_output=True, text=True, timeout=timeout)


def test_usage_and_load_failures(exe, tmp_path):
    r = run(exe)
    assert r.returncode == 1 and "Usage:" in r.stderr
    r = run(exe, tmp_path / "none.gguf", tmp_path / "a.pcm")
    assert r.returncode == 1 and "Failed to load model" in r.stderr and "cannot open" in r.stderr
    model = synth.cached_model("f32", 2, R=1)
    r = run(exe, model)                                              # no input at all
    assert r.returncode == 1 and "Usage:" in r.stderr
    r = run(exe, model, tmp_path / "missing.pcm")
    assert r.returncode == 1 and "Failed to open audio file" in r.stderr
    r = run(exe, model, "--compute", "int3", "--synthetic", "1", "1")
    assert r.returncode == 1 and "Usage:" in r.stderr
    r = run(exe, model, "--bogus")
    assert r.returncode == 1 and "unknown option" in r.stderr


def test_no_cpu_fallback(exe):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present: covered by the -m gpu tests")
    r = run(exe, synth.cached_model("f32", 2, R=1), "--right-context", "1", "--synthetic", "3", "0.5", "--gpus", "2")
    assert r.returncode == 1 and r.stdout == ""
    assert "GPU 0: Failed to load model: no CUDA device" in r.stderr and "GPU 1: Failed to load model" in r.stderr


def _oracle_tokens(path, R, pcm):
    import oracle as O
    om = O.Model(path)
    st = O.Stream(om, R)
    st.push(pcm)
    return om, st.tokens(), st.chunks


def _parse(stdout):
    rows = {}
    for line in stdout.splitlines():
        idx, name, text, toks = (line.split("\t") + [""])[:4]
        rows[int(idx)] = (name, text, [int(t) for t in toks.split()] if toks else [])
    return rows


@pytest.mark.gpu
@pytest.mark.parametrize("extra", [[], ["--realtime"], ["--warmup"]])
def test_ragged_streams_in_waves_match_the_oracle(exe, tmp_path, extra):
    """5 streams of different lengths (one shorter than a chunk, one empty) over 2 stream slots = 3 waves with slot reuse."""
    R = 1
    path = synth.cached_model("f32", 2, R=R)
    secs = [1.3, 0.9, 0.1, 2.0, 0.0]
    if extra == ["--realtime"]:
        secs = [0.7, 0.5, 0.1]                                        # real-time pacing: keep it short
    files, want = [], []
    for i, s in enumerate(secs):
        pcm = synth.synth_pcm(300 + i, s) if s > 0 else np.zeros(0, np.int16)
        f = tmp_path / f"s{i}.pcm"
        pcm.tofile(f)
        files.append(f)
        om, toks, chunks = _oracle_tokens(path, R, pcm) if s > 0 else (None, np.zeros(0, np.int32), 0)
        want.append((list(map(int, toks)), chunks))
    om = _oracle_tokens(path, R, synth.synth_pcm(300, 0.2))[0]
    lst = tmp_path / "list.txt"
    lst.write_text("\n".join(map(str, files[2:])) + "\n")
    r = run(exe, path, "--right-context", R, "--compute", "f32", "--max-streams", 2, "--tokens", *extra, files[0], files[1], "--list", lst)
    assert r.returncode == 0, r.stderr
    rows = _parse(r.stdout)
    assert sorted(rows) == list(range(len(secs)))
    for i, (toks, chunks) in enumerate(want):
        assert rows[i][0] == str(files[i])
        assert rows[i][2] == toks, (i, rows[i][2], toks)
        assert rows[i][1] == om.detok(np.asarray(toks, np.int32))
    assert f"Chunks processed:    {sum(c for _, c in want)}" in r.stderr
    assert ("Chunk latency:" in r.stderr) == (extra == ["--realtime"])


@pytest.mark.gpu
def test_flush_decodes_the_tail_like_zero_padded_audio(exe, tmp_path):
    R = 6
    path = synth.cached_model("f32", 2, R=R)
    T, n = R + 1, int(1.9 * 16000)
    pcm = synth.synth_pcm(77, 1.9)[:n]
    f = tmp_path / "a.pcm"
    pcm.tofile(f)
    plain = run(exe, path, "--right-context", R, "--compute", "f32", "--tokens", f)
    flushed = run(exe, path, "--right-context", R, "--compute", "f32", "--tokens", "--flush", f)
    assert plain.returncode == 0 and flushed.returncode == 0, plain.stderr + flushed.stderr
    frames = (n - 1) // 160 + 1
    chunks = -(-frames // (8 * T))
    padded = np.concatenate([pcm, np.zeros(1280 * T * chunks + 96 - n, np.int16)])
    _, toks_plain, c_plain = _oracle_tokens(path, R, pcm)
    _, toks_pad, c_pad = _oracle_tokens(path, R, padded)
    assert c_pad == chunks and c_pad > c_plain
    assert _parse(plain.stdout)[0][2] == list(map(int, toks_plain))
    assert _parse(flushed.stdout)[0][2] == list(map(int, toks_pad))
    assert f"Chunks processed:    {c_pad}" in flushed.stderr


@pytest.mark.gpu
def test_two_gpus_in_one_process(exe, tmp_path):
    """One process, one engine + one host thread per GPU (stream s on GPU s mod 2). Strict fp32: every stream == the oracle.
    bf16 (tcgen05 GEMMs, tensor-core attention, per-device kernel configuration): the concurrent 2-GPU run == the same streams run
    on each device alone (same batches, deterministic kernels)."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    R = 1
    path = synth.cached_model("f32", 2, R=R)
    secs = [1.3, 0.9, 1.1, 2.0, 0.6, 1.6]
    files, want = [], []
    for i, s in enumerate(secs):
        pcm = synth.synth_pcm(400 + i, s)
        f = tmp_path / f"t{i}.pcm"
        pcm.tofile(f)
        files.append(f)
        want.append(list(map(int, _oracle_tokens(path, R, pcm)[1])))
    r = run(exe, path, "--right-context", R, "--compute", "f32", "--gpus", 2, "--max-streams", 2, "--tokens", *files)
    assert r.returncode == 0, r.stderr
    assert "GPU 0: 3 streams in 2 wave(s)" in r.stderr and "GPU 1: 3 streams in 2 wave(s)" in r.stderr
    rows = _parse(r.stdout)
    for i in range(len(secs)):
        assert rows[i][2] == want[i], i
    both = run(exe, path, "--right-context", R, "--compute", "bf16", "--gpus", 2, "--tokens", *files)
    assert both.returncode == 0, both.stderr
    got = _parse(both.stdout)
    for dev in (0, 1):
        alone = run(exe, path, "--right-context", R, "--compute", "bf16", "--devices", dev, "--tokens", *files[dev::2])
        assert alone.returncode == 0, alone.stderr
        solo = _parse(alone.stdout)
        for k, i in enumerate(range(dev, len(secs), 2)):
            assert len(solo[k][2]) > 0 and solo[k][2] == got[i][2], (dev, i)


# ---------------------------------------------------------------------------------------------------------------------------
# The serve program's host loop on CPU, against a test double of the C ABI (tests/mock_nsb200.cpp: the engine's own chunk gate,
# one token = chunk index per processed chunk). Covers what the GPU cases cannot enumerate: every latency mode x ragged lengths x
# waves x GPUs x flush / realtime / warmup, with no chunk lost, duplicated or reordered.
# ---------------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def mock_exe(tmp_path_factory):
    d = tmp_path_factory.mktemp("mock")
    exe = d / "serve_mock"
    csrc = os.path.join(ROOT, "nemotron-speech.cpp_b200", "csrc")
    subprocess.check_call(["/usr/bin/g++", "-std=c++17", "-O1", "-pthread", "-I", os.path.join(ROOT, "include"), "-I", csrc,
                           os.path.join(csrc, "serve_main.cpp"), os.path.join(ROOT, "tests", "mock_nsb200.cpp"), "-o", str(exe)])
    return str(exe)


def _expected_chunks(n, T, flush):
    if flush and n > 0:
        frames = (n - 1) // 160 + 1
        return -(-frames // (8 * T))
    return max(0, (n - 96) // (1280 * T))


@pytest.mark.parametrize("R", [0, 1, 6, 13])
@pytest.mark.parametrize("mode", ["plain", "flush", "warmup", "gpus3"])
def test_serve_host_loop_on_the_mock_engine(mock_exe, tmp_path, R, mode):
    T = R + 1
    rng = np.random.default_rng(100 + R)
    lens = [0, 95, 1280 * T + 95, 1280 * T + 96, 3 * 1280 * T + 96, int(rng.integers(20000, 90000)), int(rng.integers(20000, 90000))]
    files = []
    for i, n in enumerate(lens):
        f = tmp_path / f"m{i}.pcm"
        rng.integers(-3000, 3000, n).astype(np.int16).tofile(f)
        files.append(f)
    args = [tmp_path / "model.gguf", "--right-context", R, "--tokens", "--max-streams", 3]
    args += {"plain": [], "flush": ["--flush"], "warmup": ["--warmup"], "gpus3": ["--gpus", 3, "--max-streams", 2]}[mode]
    r = run(mock_exe, *args, *files)
    assert r.returncode == 0, r.stderr
    rows = _parse(r.stdout)
    total = 0
    for i, n in enumerate(lens):
        c = _expected_chunks(n, T, mode == "flush")
        assert rows[i][2] == list(range(c)), (mode, R, i, n, rows[i][2][:5], c)       # every chunk once, in order, nothing after a reset
        total += c
    assert f"Chunks processed:    {total}\n" in r.stderr
    if mode == "gpus3":
        assert "GPU 0: 3 streams in 2 wave(s)" in r.stderr and "GPU 2: 2 streams in 1 wave(s)" in r.stderr


def test_serve_realtime_on_the_mock_engine(mock_exe, tmp_path):
    R, T = 0, 1
    lens = [16000, 9000, 12345]
    files = []
    for i, n in enumerate(lens):
        f = tmp_path / f"r{i}.pcm"; np.zeros(n, np.int16).tofile(f); files.append(f)
    r = run(mock_exe, tmp_path / "model.gguf", "--right-context", R, "--tokens", "--realtime", *files)
    assert r.returncode == 0, r.stderr
    rows = _parse(r.stdout)
    for i, n in enumerate(lens):
        assert rows[i][2] == list(range(_expected_chunks(n, T, False)))
    assert "Chunk latency:" in r.stderr and "real-time pacing" in r.stderr
    wall = float(r.stderr.split("Processing time:")[1].split("sec")[0])
    assert 0.8 <= wall <= 1.6                                            # 1 s of audio paced at audio rate


@pytest.mark.skipif(not O.reference_file("src/transcribe_stream.cpp"), reason="no reference checkout (NSB_REFERENCE_DIR)")
@pytest.mark.parametrize("R", [0, 1, 6, 13])
def test_reference_cli_on_the_shim_and_the_mock_engine(tmp_path, R):
    """The reference's own streaming CLI (byte-identical) + the drop-in shim (csrc/nemo_shim.cpp) + the test double of the C ABI, on
    CPU: the shim's push -> step-until-drained -> pop loop (nemo-stream.cpp:1074-1134) emits every chunk once and in order although
    the CLI reads 160 (9 + 8T) samples per call and a chunk consumes only 1280 T (some calls run two chunks, SURVEY appendix A);
    stdout = incremental pieces + the whole transcript + newline; stderr carries the chunk count."""
    T = R + 1
    csrc = os.path.join(ROOT, "nemotron-speech.cpp_b200", "csrc")
    src = tmp_path / "transcribe_stream.cpp"
    src.write_bytes(open(O.reference_file("src/transcribe_stream.cpp"), "rb").read())
    exe = tmp_path / "cli_mock"
    subprocess.check_call(["/usr/bin/g++", "-std=c++17", "-O1", "-I", os.path.join(ROOT, "include"), "-I", csrc, str(src),
                           os.path.join(csrc, "nemo_shim.cpp"), os.path.join(ROOT, "tests", "mock_nsb200.cpp"), "-o", str(exe)])
    n = 16000 * 9 + 777
    f = tmp_path / "a.pcm"
    np.zeros(n, np.int16).tofile(f)
    r = subprocess.run([str(exe), str(tmp_path / "model.gguf"), str(f), "70", str(R)], capture_output=True, text=True, timeout=60)
    assert r.returncode == 0, r.stderr
    chunks = _expected_chunks(n, T, False)                              # the trailing partial read is processed too (transcribe_stream.cpp:145-166)
    text = "".join(f"{c}," for c in range(chunks))
    assert r.stdout == text + text + "\n", (r.stdout[:200], chunks)
    assert f"Chunks processed:    {chunks}" in r.stderr
