"""Stream snapshots (nsb_stream_export / nsb_stream_import, include/nsb200.h; format: DESIGN.md §11), on the GPU (-m gpu).

  * strict fp32, every latency mode, four cut points (PCM only, before the ring fills, the chunk where it starts to roll, well past it)
    with steps in flight, a partial chunk buffered and tokens not yet popped: moved into another engine whose slots were used before,
    each session's tokens equal the checker's run over the whole audio, and the caches arrive bit for bit;
  * production arithmetic (bf16 / Q8_0 with the layer-ahead shadows, graph, three steps in flight): a whole engine moved into a fresh
    one -- also in permuted slot order, also onto a second GPU -- computes bit-identical tokens and encoder outputs, and the engine that
    exported continues bit-identically to one that never did;
  * round trip, the checksum recomputed here from its definition, every rejection with the error code and the field it names, and the
    edges of the C calls.
"""
import ctypes as C
import struct

import numpy as np
import pytest

import oracle as O
import synth

pytestmark = pytest.mark.gpu

HDR = 152                         # header bytes: 19 little-endian 64-bit words
W_VERSION, W_TOTAL, W_FPR, W_NL, W_R, W_KV, W_COMPUTE = 0, 1, 2, 3, 4, 5, 6
W_RING, W_VALID, W_CCPAR, W_DECPAR, W_PREV, W_CAND = 7, 8, 9, 10, 11, 12
W_BASE, W_PUSHED, W_CIDX, W_CDONE, W_NPCM, W_NTOK = 13, 14, 15, 16, 17, 18
ERR_ARG, ERR_FORMAT, ERR_STATE = -1, -3, -5
M64 = (1 << 64) - 1


def checksum(blob) -> int:
    """The snapshot checksum from its definition: sum of splitmix64(w_i + (i + 1) * golden) over the u64 words but the last."""
    w = np.frombuffer(bytes(blob), dtype="<u8")[:-1]
    with np.errstate(over="ignore"):
        z = w + (np.arange(1, len(w) + 1, dtype=np.uint64) * np.uint64(0x9E3779B97F4A7C15))
        z ^= z >> np.uint64(30); z *= np.uint64(0xBF58476D1CE4E5B9)
        z ^= z >> np.uint64(27); z *= np.uint64(0x94D049BB133111EB)
        z ^= z >> np.uint64(31)
    return int(sum(int(v) for v in z) & M64)


def word(blob, i) -> int:
    return struct.unpack_from("<q", blob, 8 * i)[0]


def stored_checksum(blob) -> int:
    return struct.unpack_from("<Q", blob, len(blob) - 8)[0]


def seal(b: bytearray) -> bytes:
    struct.pack_into("<Q", b, len(b) - 8, checksum(b))
    return bytes(b)


def with_word(blob, i, v, reseal=True) -> bytes:
    b = bytearray(blob)
    struct.pack_into("<q", b, 8 * i, v)
    return seal(b) if reseal else bytes(b)


def token_section(blob) -> np.ndarray:
    n = word(blob, W_NTOK)
    off = len(blob) - 8 - (4 * n + 7) // 8 * 8
    return np.frombuffer(blob[off:off + 4 * n], dtype="<i4")


def need(T, c):
    """raw samples that complete chunk c (host_stream.h: hs_ready)"""
    return 160 * (8 * T * (c + 1) - 1) + 256


def push_ragged(eng, s, pcm, rng):
    i = 0
    while i < len(pcm):
        k = int(rng.choice([1, 17, 333, 1500, 4000]))
        eng.push(s, pcm[i:i + k]); i += k


def caches(eng, s, n_layers=2):
    return [eng.debug_cache(s, which, layer).copy() for which in (0, 1, 2) for layer in range(n_layers)]


# ---------------------------------------------------------------------------------------------------------------------------------
# 1. strict fp32 continuation == the uninterrupted checker run, every latency mode, four cut points
# ---------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("R", [0, 1, 6, 13])
def test_strict_fp32_move_continues_like_the_uninterrupted_checker_run(built, R):
    import nsb200
    rng = np.random.default_rng(R)
    T = 1 + R
    fill = -(-70 // T)                                       # the chunk after which valid_len reaches 70 and the ring starts to roll
    cuts = [0, 2, fill, fill + 4]
    path = synth.cached_model("f32", 2, R=R)
    audio = [synth.synth_pcm(800 + 10 * R + s, (need(T, fill + 7) + 1000 + 377 * s) / 16000.0) for s in range(3)]
    om = O.Model(path)
    ref = []
    for s in range(3):
        o = O.Stream(om, R); o.push(audio[s]); ref.append((o.tokens().tolist(), o.chunks))
    A = nsb200.Engine(path, right_context=R, max_streams=3, compute=nsb200.COMPUTE_F32, cuda_graph=True)
    B = nsb200.Engine(path, right_context=R, max_streams=5, compute=nsb200.COMPUTE_F32, cuda_graph=True)
    other = [B.open_stream() for _ in range(5)]              # B's slots hold another session's state: a section the snapshot misses shows
    for k, s in enumerate(other):
        B.push(s, synth.synth_pcm(900 + k, 2.0))
    B.drain()
    for s in other:
        B.close_stream(s)
    shift = A.shift_samples
    n_tok = 0
    for c in cuts:
        ids = [A.open_stream() for _ in range(3)]
        popped = [[] for _ in range(3)]
        pushed = [0] * 3
        for s in range(3):
            pushed[s] = need(T, 0) - 1 - 100 * s if c == 0 else need(T, c - 1) + 17 + s * (shift // 3)   # + a partial chunk
            push_ragged(A, ids[s], audio[s][:pushed[s]], rng)
        n_plain = max(0, c - 3)
        for i in range(n_plain):
            assert A.step() == 3
            if i % 2 == 0:
                for s in range(3):
                    popped[s] += A.pop_tokens(ids[s]).tolist()
        for i in range(c - n_plain):                         # up to three steps in flight at the export
            assert A.step_begin() == 3
        assert not any(A.ready(i) for i in ids)
        blobs = [A.export_stream(i) for i in ids]
        for s, b in enumerate(blobs):
            assert b[:4] == b"NSBS" and word(b, W_TOTAL) == len(b) and stored_checksum(b) == checksum(b)
            assert word(b, W_CIDX) == word(b, W_CDONE) == c and word(b, W_PUSHED) == pushed[s]
            assert word(b, W_VALID) == min(70, T * c) and word(b, W_RING) == (T * c) % (70 + T)
        before = [caches(A, i) for i in ids]
        for s, i in enumerate(ids):                          # the queued tokens are in the snapshot and stay poppable on the stream
            assert np.array_equal(A.pop_tokens(i), token_section(blobs[s]))
            assert A.chunks(i) == c
            A.close_stream(i)
        slots = [B.import_stream(b) for b in blobs]
        assert slots == [0, 1, 2]
        for s in range(3):
            after = caches(B, slots[s])
            for k in range(len(after)):
                assert np.array_equal(after[k].view(np.uint32), before[s][k].view(np.uint32)), (c, s, k)
            assert B.export_stream(slots[s]) == blobs[s]     # round trip, byte for byte
            assert B.chunks(slots[s]) == c
        # the rest of the audio, in ragged pieces, stepped in a random mix of plain and split steps
        rest = [[] for _ in range(3)]
        inflight = 0
        while any(pushed[s] < len(audio[s]) for s in range(3)):
            for s in range(3):
                k = int(rng.choice([1, 17, shift // 3, shift, 2 * shift]))
                piece = audio[s][pushed[s]:pushed[s] + k]
                if len(piece):
                    B.push(slots[s], piece); pushed[s] += len(piece)
            if rng.random() < 0.4:
                while inflight:
                    B.step_end(); inflight -= 1
                B.step()
            else:
                while inflight < 3 and B.step_begin() > 0:
                    inflight += 1
                if inflight and rng.random() < 0.7:
                    B.step_end(); inflight -= 1
            for s in range(3):
                rest[s] += B.pop_tokens(slots[s]).tolist()
        while inflight:
            B.step_end(); inflight -= 1
        B.drain()
        for s in range(3):
            rest[s] += B.pop_tokens(slots[s]).tolist()
            assert popped[s] + rest[s] == ref[s][0], (R, c, s)
            assert B.chunks(slots[s]) == ref[s][1], (R, c, s)
            n_tok += len(rest[s])
            B.close_stream(slots[s])
    assert n_tok > 30
    A.close(); B.close()


# ---------------------------------------------------------------------------------------------------------------------------------
# 2./3./7. production arithmetic: a whole engine moved is bit-identical; the exporting engine is undisturbed
# ---------------------------------------------------------------------------------------------------------------------------------
def move_whole_engine(wtype, compute, kv, R, n, k_steps, permute, device_b=0):
    """Engines A (exports), C (control, never exports) and B (imports A's streams after k steps), all driven with the same pushes and
    the same schedule of three steps in flight: after the move, A, B and C must compute the same tokens and encoder outputs bit for bit."""
    import nsb200
    path = synth.cached_model(wtype, 2, R=R)
    T = 1 + R
    mk = lambda dev: nsb200.Engine(path, right_context=R, max_streams=n, compute=compute, kv_dtype=kv, cuda_graph=True, decode_overlap=0,
                                   device=dev)
    A, C = mk(0), mk(0)
    chunks = k_steps + 9
    L = need(T, chunks - 1) + 100
    audio = np.stack([synth.synth_pcm(700 + s, L / 16000.0 + 0.01)[:L] for s in range(n)])
    ids = {id(A): np.array([A.open_stream() for _ in range(n)], np.int32), id(C): np.array([C.open_stream() for _ in range(n)], np.int32)}
    shift, pos = A.shift_samples, 0
    engines = [A, C]
    toks = {id(A): [[] for _ in range(n)], id(C): [[] for _ in range(n)]}

    def feed(k):
        nonlocal pos
        if pos < L:
            for e in engines:
                e.push_batch(ids[id(e)], audio[:, pos:pos + k])
            pos += k

    def x_by_stream(e):                                        # rows are in slot order; reorder to stream order
        x = e.debug_get("x", n).reshape(n, T, 1024)
        order = np.argsort(np.argsort(ids[id(e)]))             # stream i sits at batch row rank(slot of i)
        return x[order]

    def pop_all():
        for e in engines:
            t, cnt = e.pop_tokens_batch(ids[id(e)], 64 * T)
            for s in range(n):
                toks[id(e)][s] += t[s, :cnt[s]].tolist()

    def run(steps):
        """steps = None: until the audio is used up; otherwise return after that many step_end, with three steps in flight"""
        inflight = done = 0
        while True:
            while inflight < 3:
                nb = [e.step_begin() for e in engines]
                assert len(set(nb)) == 1 and nb[0] in (0, n), nb
                if nb[0] == 0:
                    break
                x0 = x_by_stream(engines[0])
                for e in engines[1:]:
                    assert np.array_equal(x_by_stream(e).view(np.uint32), x0.view(np.uint32))
                inflight += 1
                feed(shift)
            if done == steps or inflight == 0:
                return inflight
            for e in engines:
                assert e.step_end() == n
            inflight -= 1; done += 1
            pop_all()

    feed(need(T, 0))
    inflight = run(k_steps)
    assert inflight == 3
    blobs = [A.export_stream(int(i)) for i in ids[id(A)]]      # collects A's steps in flight; C collects the same steps below
    for _ in range(inflight):
        assert C.step_end() == n
    assert A.step_end() == 0
    B = mk(device_b)
    order = np.random.default_rng(n).permutation(n) if permute else np.arange(n)
    slot_b = np.empty(n, np.int32)
    for j, s in enumerate(order):
        slot_b[s] = B.import_stream(blobs[s])
        assert slot_b[s] == j
    ids[id(B)] = slot_b
    toks[id(B)] = [list(t) for t in toks[id(A)]]               # tokens popped before the move
    engines = [C, A, B]
    pop_all()
    run(None)
    pop_all()
    for s in range(n):
        assert toks[id(A)][s] == toks[id(C)][s] == toks[id(B)][s], s
        assert A.chunks(int(ids[id(A)][s])) == B.chunks(int(slot_b[s])) == C.chunks(int(ids[id(C)][s])) == chunks
    assert sum(len(t) for t in toks[id(C)]) > 5 * n
    for e in engines:
        e.close()


@pytest.mark.parametrize("wtype,compute,kv,R,n,k_steps,permute", [
    ("f16", 3, 2, 1, 64, 10, False),                           # BASELINE.json config 2's arithmetic: bf16 GEMMs, bf16 K/V
    ("q8_0", 0, 1, 6, 16, 4, False),                           # Q8_0 file: fp16 layer-ahead shadows of the quantised matrices
    ("f16", 3, 2, 1, 64, 10, True),                            # streams land in other slots
], ids=["bf16_R1_64", "q8_0_R6_16", "bf16_R1_64_permuted"])
def test_moving_a_whole_engine_is_bit_identical(built, wtype, compute, kv, R, n, k_steps, permute):
    move_whole_engine(wtype, compute, kv, R, n, k_steps, permute)


def test_moving_a_whole_engine_to_another_gpu_is_bit_identical(built):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    move_whole_engine("f16", 3, 2, 1, 64, 10, True, device_b=1)


# ---------------------------------------------------------------------------------------------------------------------------------
# 5. rejection: malformed blobs (NSB_ERR_FORMAT) and incompatible engines (NSB_ERR_ARG), nothing changed after any of them
# ---------------------------------------------------------------------------------------------------------------------------------
def expect_reject(eng, blob, code, field):
    """No step runs between a crafted import and this check; a blob that is wrongly accepted is closed again before failing."""
    import nsb200
    try:
        s = eng.import_stream(blob)
    except nsb200.NsbError as e:
        msg = str(e)
        assert msg.startswith(f"nsb error {code}:") and field in msg, (code, field, msg)
        return
    eng.close_stream(s)
    pytest.fail(f"snapshot accepted, expected error {code} naming {field!r}")


def test_rejected_snapshots_change_nothing(built):
    import nsb200
    R, T = 1, 2
    path = synth.cached_model("f32", 2, R=R)
    om = O.Model(path)
    mk = lambda **kw: nsb200.Engine(path, **{"right_context": R, "max_streams": 3, "compute": nsb200.COMPUTE_F32, **kw})
    A = mk()
    pcm = synth.synth_pcm(950, 3.0)
    s = A.open_stream()
    cut = need(T, 5) + 500
    A.push(s, pcm[:cut]); A.drain()
    blob = A.export_stream(s)
    assert word(blob, W_NTOK) > 0 and word(blob, W_NPCM) > 0
    A.close()
    # B: one live stream that must continue bit-identically (= the checker's tokens, strict fp32) through every rejection
    B = mk()
    live_pcm = synth.synth_pcm(951, 3.0)
    live = B.open_stream()
    B.push(live, live_pcm[:need(T, 3) + 99]); B.step(); B.step_begin(); B.step_begin()
    kv_bytes = 2 * 2 * (70 + T) * 1024 * 4
    tok_off = len(blob) - 8 - (4 * word(blob, W_NTOK) + 7) // 8 * 8

    def bit(b, off, k=1):
        b = bytearray(b); b[off] ^= k; return bytes(b)

    def tok5000():
        b = bytearray(blob); struct.pack_into("<i", b, tok_off, 5000); return seal(b)

    malformed = [
        (blob[:HDR + 8], "size"), (blob[:HDR + kv_bytes // 2], "size"), (blob[:-1], "size"), (blob[:HDR - 8], "size"),
        (b"X" + blob[1:], "magic"), (with_word(blob, W_VERSION, word(blob, W_VERSION) + (1 << 32)), "version"),
        (bit(blob, 8 * W_FPR + 3, 0x20), "checksum"), (bit(blob, 8 * W_DECPAR), "checksum"), (bit(blob, 8 * W_CAND), "checksum"),
        (bit(blob, HDR + 1001, 0x10), "checksum"), (bit(blob, len(blob) - 1, 0x80), "checksum"),
        (with_word(blob, W_RING, 70 + T), "ring_pos"), (with_word(blob, W_PREV, 1025), "prev_token"), (with_word(blob, W_DECPAR, 2), "dec_par"),
        (with_word(blob, W_CCPAR, 2), "cc_par"), (with_word(blob, W_VALID, 71), "valid_len"), (with_word(blob, W_CAND, 2), "cand_valid"),
        (with_word(blob, W_BASE, word(blob, W_BASE) + 1), "base"), (with_word(blob, W_CDONE, word(blob, W_CDONE) - 1), "chunks_done"),
        (tok5000(), "token id"),
    ]
    for b, field in malformed:
        expect_reject(B, b, ERR_FORMAT, field)
        nxt = B.open_stream()                                  # no slot was consumed
        assert nxt == 1, (field, nxt)
        B.close_stream(nxt)
    # a valid import after all that: slot 1, and both streams continue like the checker
    moved = B.import_stream(blob)
    assert moved == 1
    B.push(live, live_pcm[need(T, 3) + 99:]); B.push(moved, pcm[cut:])
    B.drain()
    for sid, audio in ((live, live_pcm), (moved, pcm)):
        o = O.Stream(om, R); o.push(audio)
        assert np.array_equal(B.pop_tokens(sid), o.tokens()) and B.chunks(sid) == o.chunks
    B.close()
    # incompatible engines: a valid snapshot that does not fit is an argument error naming the field
    for kw, field, p in [({"right_context": 6}, "att_right_context", path), ({"kv_dtype": nsb200.KV_F16}, "kv_dtype", path),
                         ({"compute": nsb200.COMPUTE_F16}, "compute", path),
                         ({}, "n_layers", synth.cached_model("f32", 3, R=R)), ({}, "fingerprint", synth.cached_model("f32", 2, seed=77, R=R))]:
        E = nsb200.Engine(p, **{"right_context": R, "max_streams": 2, "compute": nsb200.COMPUTE_F32, **kw})
        expect_reject(E, blob, ERR_ARG, field)
        assert E.open_stream() == 0
        E.close()


# ---------------------------------------------------------------------------------------------------------------------------------
# 6. API edges
# ---------------------------------------------------------------------------------------------------------------------------------
def test_export_import_api_edges(built, tmp_path):
    import shutil
    import nsb200
    R, T = 1, 2
    path = synth.cached_model("f32", 2, R=R)
    om = O.Model(path)
    L = nsb200.lib()
    A = nsb200.Engine(path, right_context=R, max_streams=2, compute=nsb200.COMPUTE_F32)
    pcm = synth.synth_pcm(960, 2.5)
    s = A.open_stream()
    cut = need(T, 4) + 1234
    A.push(s, pcm[:cut]); A.step(); A.step_begin(); A.step_begin()
    n = int(L.nsb_stream_export(A.h, s, None, 0))              # collects the two steps in flight, then sizes the snapshot
    buf = C.create_string_buffer(b"\xab" * n, n)
    assert int(L.nsb_stream_export(A.h, s, buf, n - 1)) == ERR_ARG and "needs" in L.nsb_last_error().decode()
    assert buf.raw == b"\xab" * n                              # untouched
    assert int(L.nsb_stream_export(A.h, s, buf, n)) == n and stored_checksum(buf.raw) == checksum(buf.raw)
    blob = buf.raw
    assert A.export_stream(s) == blob                         # nothing ran in between: the same bytes
    for bad in (1, -1, 2, 99):                                 # closed, invalid, the batch path's private slot, invalid
        assert int(L.nsb_stream_export(A.h, bad, buf, n)) == ERR_ARG
    # a full engine: NSB_ERR_STATE, and nothing changed
    full = A.open_stream()
    A.push(full, pcm[:5000])
    before = A.export_stream(full)
    expect_reject(A, blob, ERR_STATE, "no free stream slot")
    assert A.export_stream(full) == before and A.export_stream(s) == blob
    A.close()
    # the snapshot outlives its engine, and the same model file at another path has the same fingerprint
    copy = str(tmp_path / "same_model.gguf")
    shutil.copyfile(path, copy)
    B = nsb200.Engine(copy, right_context=R, max_streams=1, compute=nsb200.COMPUTE_F32)
    s2 = B.import_stream(blob)
    assert s2 == 0
    B.push(s2, pcm[cut:]); B.drain()
    o = O.Stream(om, R); o.push(pcm)
    assert np.array_equal(B.pop_tokens(s2), o.tokens()) and B.chunks(s2) == o.chunks
    B.close()
