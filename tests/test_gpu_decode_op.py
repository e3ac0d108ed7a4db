"""Operator tests of the RNN-T greedy-decode kernel (rnnt_decode_kernel, csrc/kernels_decode.cu) against float64, through
nsb_op_decode (include/nsb200.h): the step's own launch on the engine's decoder weights, with state and outputs private to the call.

The kernel runs the same arithmetic through eight device code paths, chosen per phase from the grid size and the number of streams
in the round (phase_dispatch): phase<RPL, 1 | 2>, phase_pipe<1,1>, <1,2>, <1,4>, <2,4> and phase_gemv<1 | 2>. All of them sum K in
the same eight chunks in the same order, so every launch of the same inputs must give the same bits. The tests check:
  * bit identity of tokens, frames, counts, the final state of every slot and the logits of batch row 0 across six launches (full
    grid, full grid with the pipelined tiles from one stream on, 20, 2 and 64 CTA pairs, and a plain 96-CTA grid), with a Python
    mirror of phase_dispatch asserting which templates each case reached and that the cases together reach all eight;
  * every decision against a float64 reference run TEACHER-FORCED (it takes the kernel's decisions, so a near-tie cannot make the
    two runs diverge): the chosen token's float64 logit is within BOUND_LOGIT x scale of the float64 maximum, and the token is the
    float64 argmax whenever the top-2 gap exceeds that; scale = max over the vocabulary of |relu(enc + dec)| . |w_v| + |b_v|;
  * row 0's token at every evaluation == the first argmax of its own fp32 logits (the cross-CTA key, no tolerance), and those
    logits against float64;
  * counts, frames, prev_token, par and cand_valid exactly, the committed and candidate h / c and dec_proj against float64, and
    every slot outside the batch bit for bit unchanged;
  * the symbol cap (10 per frame, no blank evaluation after the tenth, the 10 T output buffer full and its guards untouched), exact
    ties (duplicated rows of joint.joint_net.2: the lower index wins, a token tied with blank emits) and argument errors.
Frames are forced with enc_proj = ALPHA * joint_net.2 row: towards blank (1 evaluation per frame) or towards a token (10 emissions).
With NSB_DECODE_OPS_REPORT=<file> set, every case appends its measured maxima as one JSON line: the data the bounds are set from.
"""
import ctypes as C
import json
import os
import shutil

import numpy as np
import pytest

import synth

BLANK, VOCAB, HID, MAX_SYMBOLS = 1024, 1025, 640, 10
ALPHA = 40.0                    # forced frames: logit of the target ~ ALPHA / 2, the rest within a few units
# Bounds, each 2x - 3.5x above the largest value measured over every case of its class on an NVIDIA B200 (1000 W power limit).
BOUND_LOGIT = 6e-7              # |logit - float64| / scale (row 0), and the float64 shortfall of a chosen token: measured 2.4e-7 (T = 2048), shortfall 0
BOUND_STATE = 1e-5              # |x - float64| / (|x| + 1) over h, c, dec_proj: measured 3.4e-6 (carried state, B = 130)

LAUNCHES = {"full": (0, 0), "full_pipe1": (0, 1), "narrow20": (20, 0), "narrow2": (2, 0), "narrow64": (64, 0), "plain96": (96, 0)}
# phase<n> = phase<RPL, n> (RPL = 5 for the LSTM, 2 otherwise), pipe<r,s> = phase_pipe<r, s>, gemv<n> = phase_gemv<n>
ALL_TEMPLATES = {"phase<1>", "phase<2>", "pipe<1,1>", "pipe<1,2>", "pipe<1,4>", "pipe<2,4>", "gemv<1>", "gemv<2>"}
PIPE_MIN_N = 65                 # launch_decode's default


def report(**kw):
    path = os.environ.get("NSB_DECODE_OPS_REPORT")
    if path:
        with open(path, "a") as f:
            f.write(json.dumps(kw) + "\n")


# ------------------------------------------------------------------------------------------------------------------------------
# float64 reference (torch, on the CPU for the unmarked tests and on the GPU for the operator tests)
# ------------------------------------------------------------------------------------------------------------------------------
class Ref:
    """The decoder's weights in float64 and the three operations of one evaluation."""

    def __init__(self, path, device="cpu"):
        import torch
        import nsb200
        self.dev = device
        t = lambda n, shape: torch.from_numpy(nsb200.read_tensor(path, n)[0].reshape(shape).astype(np.float64)).to(device)
        d = "decoder.prediction."
        self.embed = t(d + "embed.weight", (VOCAB, HID))
        self.w_ih = [t(d + f"dec_rnn.lstm.weight_ih_l{l}", (4 * HID, HID)) for l in range(2)]
        self.w_hh = [t(d + f"dec_rnn.lstm.weight_hh_l{l}", (4 * HID, HID)) for l in range(2)]
        self.b_ih = [t(d + f"dec_rnn.lstm.bias_ih_l{l}", (4 * HID,)) for l in range(2)]
        self.b_hh = [t(d + f"dec_rnn.lstm.bias_hh_l{l}", (4 * HID,)) for l in range(2)]
        self.pred_w, self.pred_b = t("joint.pred.weight", (HID, HID)), t("joint.pred.bias", (HID,))
        self.out_w, self.out_b = t("joint.joint_net.2.weight", (VOCAB, HID)), t("joint.joint_net.2.bias", (VOCAB,))
        self.enc_w, self.enc_b = t("joint.enc.weight", (HID, 1024)), t("joint.enc.bias", (HID,))
        self.abs_out_w, self.abs_out_b = self.out_w.abs(), self.out_b.abs()

    def lstm(self, l, x, h, c):
        """one LSTM layer, gate order i, f, g, o: [n, 640] each"""
        import torch
        g = x @ self.w_ih[l].T + h @ self.w_hh[l].T + self.b_ih[l] + self.b_hh[l]
        i, f, gg, o = g.split(HID, dim=1)
        c2 = torch.sigmoid(f) * c + torch.sigmoid(i) * torch.tanh(gg)
        return torch.sigmoid(o) * torch.tanh(c2), c2

    def candidate(self, prev, h, c):
        """(h', c' [n, 1280], joint.pred projection [n, 640]) for previous tokens prev [n] and committed h, c [n, 1280]"""
        import torch
        h0, c0 = self.lstm(0, self.embed[prev], h[:, :HID], c[:, :HID])
        h1, c1 = self.lstm(1, h0, h[:, HID:], c[:, HID:])
        return torch.cat([h0, h1], 1), torch.cat([c0, c1], 1), h1 @ self.pred_w.T + self.pred_b

    def logits(self, enc, dec):
        """(logits [n, 1025], scale [n]) of the joint relu(enc + dec) . joint_net.2"""
        z = (enc + dec).clamp_min(0.0)
        return z @ self.out_w.T + self.out_b, (z @ self.abs_out_w.T + self.abs_out_b).amax(1)


class State64:
    """float64 decoder state of n streams, updated like the kernel's slots: blank leaves it alone, an emission commits the
    candidate and invalidates it. `old_*` is the committed state before the last emission (the kernel's other parity buffer)."""

    def __init__(self, ref, h, c, cand_h, cand_c, dec_proj, valid, prev):
        import torch
        f = lambda a: torch.as_tensor(np.asarray(a, dtype=np.float64), device=ref.dev).clone()
        self.ref, self.h, self.c, self.ch, self.cc, self.proj = ref, f(h), f(c), f(cand_h), f(cand_c), f(dec_proj)
        self.old_h, self.old_c = self.ch.clone(), self.cc.clone()
        self.valid = torch.as_tensor(np.asarray(valid, dtype=bool), device=ref.dev).clone()
        self.prev = torch.as_tensor(np.asarray(prev, dtype=np.int64), device=ref.dev).clone()
        self.emitted = np.zeros(len(prev), dtype=np.int64)

    def evaluate(self, idx, enc):
        """logits and scale of streams idx (numpy int array) on enc rows [len(idx), 640]; refreshes stale candidates first"""
        import torch
        ti = torch.as_tensor(idx, device=self.ref.dev)
        stale = ti[~self.valid[ti]]
        if len(stale):
            self.ch[stale], self.cc[stale], self.proj[stale] = self.ref.candidate(self.prev[stale], self.h[stale], self.c[stale])
            self.valid[stale] = True
        return self.ref.logits(enc, self.proj[ti])

    def apply(self, idx, tok):
        """decisions tok (numpy) of streams idx"""
        import torch
        e = idx[tok != BLANK]
        if len(e):
            te = torch.as_tensor(e, device=self.ref.dev)
            self.old_h[te], self.old_c[te] = self.h[te], self.c[te]
            self.h[te], self.c[te] = self.ch[te], self.cc[te]
            self.prev[te] = torch.as_tensor(tok[tok != BLANK], device=self.ref.dev)
            self.valid[te] = False
            self.emitted[e] += 1


def greedy64(st, enc_proj):
    """free-running float64 greedy decode of ONE stream over enc_proj [T, 640] (torch) -> (tokens, [(logits, scale)] per
    evaluation); at most MAX_SYMBOLS emissions per frame, the lowest index among the maxima"""
    import torch
    toks, evals, i0 = [], [], np.array([0])
    for t in range(enc_proj.shape[0]):
        for _ in range(MAX_SYMBOLS):
            lg, sc = st.evaluate(i0, enc_proj[t:t + 1])
            evals.append((lg[0], float(sc[0])))
            tok = int(torch.argmax(lg[0]))                                    # first occurrence of the maximum
            st.apply(i0, np.array([tok]))
            if tok == BLANK:
                break
            toks.append(tok)
    return toks, evals


def fresh_state(S):
    """the engine's state of a freshly opened slot, S slots"""
    z = np.zeros((S, 2, 2 * HID), np.float32)
    return dict(h=z, c=z.copy(), dec_proj=np.zeros((S, HID), np.float32), par=np.zeros(S, np.int32),
                prev_token=np.full(S, BLANK, np.int32), cand_valid=np.zeros(S, np.int32))


# ------------------------------------------------------------------------------------------------------------------------------
# CPU tests of the reference
# ------------------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ref_cpu(built):
    return Ref(synth.cached_model("f32", 2, R=0))


def test_lstm_step_matches_torch_lstm(ref_cpu):
    """Ref.candidate's two LSTM layers == torch.nn.LSTM with the file's weights (gate order i, f, g, o)"""
    import torch
    ref = ref_cpu
    lstm = torch.nn.LSTM(HID, HID, num_layers=2).double()
    with torch.no_grad():
        for l in range(2):
            getattr(lstm, f"weight_ih_l{l}").copy_(ref.w_ih[l]); getattr(lstm, f"weight_hh_l{l}").copy_(ref.w_hh[l])
            getattr(lstm, f"bias_ih_l{l}").copy_(ref.b_ih[l]); getattr(lstm, f"bias_hh_l{l}").copy_(ref.b_hh[l])
    rng = np.random.default_rng(3)
    n = 5
    prev = torch.as_tensor(rng.integers(0, VOCAB, n))
    h = torch.as_tensor(np.tanh(rng.standard_normal((n, 2 * HID))))
    c = torch.as_tensor(rng.standard_normal((n, 2 * HID)))
    h1, c1, proj = ref.candidate(prev, h, c)
    with torch.no_grad():
        y, (hn, cn) = lstm(ref.embed[prev][None], (h.reshape(n, 2, HID).transpose(0, 1).contiguous(),
                                                   c.reshape(n, 2, HID).transpose(0, 1).contiguous()))
    assert torch.allclose(h1, hn.transpose(0, 1).reshape(n, 2 * HID), rtol=0, atol=1e-12)
    assert torch.allclose(c1, cn.transpose(0, 1).reshape(n, 2 * HID), rtol=0, atol=1e-12)
    assert torch.allclose(proj, y[0] @ ref.pred_w.T + ref.pred_b, rtol=0, atol=1e-12)


def test_reference_greedy_matches_cpu_checker(ref_cpu):
    """float64 joint.enc on the checker's encoder output, then greedy64 with the decoder state carried from chunk to chunk:
    the checker's tokens, and its logits at every evaluation (up to a near-tie of the checker's fp32 arithmetic)"""
    import torch
    import oracle as O
    ref, R = ref_cpu, 1
    om = O.Model(synth.cached_model("f32", 2, R=0))
    o = O.Stream(om, R, trace=True)
    o.push(synth.synth_pcm(7, 2.5))
    assert o.chunks >= 10
    st = State64(ref, *(np.zeros((1, 2 * HID)),) * 4, np.zeros((1, HID)), [False], [BLANK])
    toks, evals = [], []
    for ch in range(o.chunks):
        x = torch.as_tensor(o.trace_enc(ch).astype(np.float64))
        t, e = greedy64(st, x @ ref.enc_w.T + ref.enc_b)
        toks += t; evals += e
    want = o.tokens()
    assert len(want) >= 10 and o.n_evals() >= 30, (len(want), o.n_evals())
    n = min(len(evals), o.n_evals())
    for ev in range(n):
        lo = torch.as_tensor(o.trace_logits(ev).astype(np.float64))
        lg, sc = evals[ev]
        assert float((lo - lg).abs().max()) <= 1e-5 * sc, ev
        if o.eval_token(ev) != int(torch.argmax(lg)):                     # a near-tie: the rest of the two runs differ
            top = torch.topk(lg, 2).values
            assert float(top[0] - top[1]) <= 2e-5 * sc, ev
            return
    assert toks == list(want)
    assert len(evals) == o.n_evals()


# ------------------------------------------------------------------------------------------------------------------------------
# GPU side
# ------------------------------------------------------------------------------------------------------------------------------
_engines, _refs = {}, {}


def _tie_model(dst_dir):
    """the synthetic f32 model with rows of joint.joint_net.2 (weights and bias) duplicated: 17 := 16 (one 8-row item, one
    32-row tile), 1000 := 3 (different CTAs), 500 := 1024 (a token that ties with blank: it always wins, blank never does)"""
    src = synth.cached_model("f32", 2, R=0)
    dst = os.path.join(dst_dir, "tie_f32_L2.gguf")
    shutil.copyfile(src, dst)
    header, infos = synth._gguf_header(2, "f32", 1234)
    where = {name: (len(header) + off, nbytes) for name, _, _, off, nbytes in infos}
    with open(dst, "r+b") as f:
        for name, width in (("joint.joint_net.2.weight", HID), ("joint.joint_net.2.bias", 1)):
            off, nbytes = where[name]
            f.seek(off)
            a = np.frombuffer(f.read(nbytes), dtype=np.float32).reshape(VOCAB, width).copy()
            for dst_row, src_row in TIE_PAIRS:
                a[dst_row] = a[src_row]
            f.seek(off)
            f.write(a.tobytes())
    return dst


TIE_PAIRS = ((17, 16), (1000, 3), (500, 1024))


@pytest.fixture(scope="module")
def dec(built, tmp_path_factory):
    """kind ('plain' | 'tie') -> (engine, float64 reference on the GPU)"""
    import nsb200

    def get(kind):
        if kind not in _engines:
            path = synth.cached_model("f32", 2, R=0) if kind == "plain" else _tie_model(str(tmp_path_factory.mktemp("tie")))
            _engines[kind] = nsb200.Engine(path, right_context=0, max_streams=1, compute=nsb200.COMPUTE_F32)
            _refs[kind] = Ref(path, "cuda")
        return _engines[kind], _refs[kind]
    yield get
    for e in _engines.values():
        e.close()
    _engines.clear(); _refs.clear()


def sm_count():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def natural_frames(ref, shape, rng):
    """enc_proj rows like joint.enc's on this model: joint.enc of encoder rows that deviate from their mean by 0.4 N(0, 1) (the
    calibrated joint.enc bias cancels the mean), plus the bias's own 0.1 N(0, 1). About one frame in six starts an emission."""
    n = int(np.prod(shape))
    x = 0.4 * rng.standard_normal((n, 1024)) @ ref.enc_w.cpu().numpy().T + 0.1 * rng.standard_normal((n, HID))
    return x.astype(np.float32).reshape(*shape, HID)


def forced(ref, tok):
    """an enc_proj row that drives the joint towards tok: ALPHA * joint_net.2 row tok"""
    return (ALPHA * ref.out_w[tok].cpu().numpy()).astype(np.float32)


def inputs(ref, B, T, rng, S=None, frac_forced=0.0):
    """enc_proj of natural frames, a fraction of them forced towards blank or a random token; fresh state; identity slot map"""
    enc = natural_frames(ref, (B, T), rng)
    for b, t in zip(*np.nonzero(rng.random((B, T)) < frac_forced)):
        enc[b, t] = forced(ref, BLANK if rng.random() < 0.5 else int(rng.integers(0, BLANK)))
    S = S or B
    return dict(enc_proj=enc, slot_of_b=np.arange(B, dtype=np.int32), **fresh_state(S))


def run(eng, inp, launch):
    grid, pipe = LAUNCHES[launch]
    out = eng.op_decode(inp["enc_proj"], inp["h"], inp["c"], inp["dec_proj"], inp["par"], inp["prev_token"], inp["cand_valid"],
                        inp["slot_of_b"], grid=grid, pipe_min_n=pipe)
    assert out["guard_bad"] == 0, f"{out['guard_bad']} guard entries written"
    assert out["grid_used"] == (grid or sm_count()), out["grid_used"]
    return out


def decisions(out, T):
    """per batch row, the kernel's decision at each joint evaluation, rebuilt from its tokens and frames: the frame's tokens, then
    a blank unless the frame reached MAX_SYMBOLS -> (list of (frame, decision) lists, emissions per frame [B, T])"""
    B = out["counts"].shape[0]
    seqs, per_frame = [], np.zeros((B, T), np.int64)
    for b in range(B):
        n = int(out["counts"][b])
        assert 0 <= n <= MAX_SYMBOLS * T, n
        tk, fr = out["tokens"][b, :n], out["frames"][b, :n]
        assert np.all(out["tokens"][b, n:] == -1) and np.all(out["frames"][b, n:] == -1), "entries past the count were written"
        assert np.all((tk >= 0) & (tk < BLANK)), "a blank or out-of-range token was emitted"
        assert np.all((fr >= 0) & (fr < T)) and np.all(np.diff(fr) >= 0), "frames out of order"
        per_frame[b] = np.bincount(fr, minlength=T)
        assert per_frame[b].max(initial=0) <= MAX_SYMBOLS
        s, i = [], 0
        for t in range(T):
            k = int(per_frame[b, t])
            s += [(t, int(v)) for v in tk[i:i + k]]
            i += k
            if k < MAX_SYMBOLS:
                s.append((t, BLANK))
        seqs.append(s)
    return seqs, per_frame


def round_counts(seqs, cand_valid0):
    """(streams with a stale candidate, active streams) per round, as the kernel's compaction sees them"""
    E = max(len(s) for s in seqs)
    need, act = [], []
    for r in range(E):
        a = [b for b, s in enumerate(seqs) if r < len(s)]
        act.append(len(a))
        need.append(sum(1 for b in a if (seqs[b][r - 1][1] != BLANK if r else not cand_valid0[b])))
    return need, act


def templates(launch, need, act):
    """the device templates phase_dispatch picks for these rounds (a mirror of phase_dispatch)"""
    grid, pipe_min_n = LAUNCHES[launch]
    grid, pipe_min_n = grid or sm_count(), pipe_min_n or PIPE_MIN_N
    narrow, got = grid <= 64, set()
    for mode, ns in (("lstm", need), ("pred", need), ("joint", act)):
        for n in ns:
            if n == 0:
                continue
            if not (narrow or n >= pipe_min_n):
                got.add("phase<1>" if n <= 8 else "phase<2>")
            elif narrow and mode == "lstm" and n <= 16:
                got.add("gemv<1>" if n <= 8 else "gemv<2>")
            elif narrow and mode == "joint" and n > 16:
                got.add("pipe<2,4>")
            else:
                got.add("pipe<1,1>" if n <= 8 else "pipe<1,2>" if n <= 16 else "pipe<1,4>" if n <= 64 else "pipe<2,4>")
    return got


def assert_same(a, b, what):
    for k in ("tokens", "frames", "counts", "par", "prev_token", "cand_valid", "n_logits"):
        assert np.array_equal(a[k], b[k]), f"{what}: {k} differs"
    for k in ("h", "c", "dec_proj", "logits"):
        assert np.array_equal(a[k].view(np.uint32), b[k].view(np.uint32)), f"{what}: {k} differs in bits"


def check_row0(out, seqs):
    """batch row 0: one tapped logit row per evaluation, and its decision is exactly the first argmax of that row"""
    lg = out["logits"]
    assert out["n_logits"] == len(seqs[0]) and lg.shape[0] == len(seqs[0])
    assert np.isfinite(lg).all()
    got = [d for _, d in seqs[0]]
    want = np.argmax(lg, axis=1).tolist()
    assert got == want, [(i, g, w) for i, (g, w) in enumerate(zip(got, want)) if g != w][:5]


def check_f64(ref, inp, out, seqs, rows):
    """teacher-forced float64 check of batch rows `rows` (module docstring) -> measured maxima"""
    import torch
    rows = np.asarray(rows)
    slots = inp["slot_of_b"][rows]
    par0 = inp["par"][slots]
    pick = lambda a, p: a[slots, p]
    st = State64(ref, pick(inp["h"], par0), pick(inp["c"], par0), pick(inp["h"], 1 - par0), pick(inp["c"], 1 - par0),
                 inp["dec_proj"][slots], inp["cand_valid"][slots] == 1, inp["prev_token"][slots])
    enc = torch.as_tensor(inp["enc_proj"][rows].astype(np.float64), device=ref.dev)
    n = len(rows)
    E = np.array([len(seqs[b]) for b in rows])
    worst = dict(logit=0.0, gap=0.0, state=0.0)
    tap = out["logits"]
    row0 = np.nonzero(rows == 0)[0]
    for r in range(int(E.max())):
        idx = np.nonzero(E > r)[0]
        fr = np.array([seqs[rows[i]][r][0] for i in idx])
        dec = np.array([seqs[rows[i]][r][1] for i in idx])
        lg, sc = st.evaluate(idx, enc[torch.as_tensor(idx, device=ref.dev), torch.as_tensor(fr, device=ref.dev)])
        mx = lg.max(1).values
        chosen = lg.gather(1, torch.as_tensor(dec, device=ref.dev)[:, None])[:, 0]
        gap = ((mx - chosen) / sc).cpu().numpy()
        worst["gap"] = max(worst["gap"], float(gap.max()))
        assert gap.max() <= BOUND_LOGIT, ("a token below the float64 maximum", r, rows[idx[gap.argmax()]], float(gap.max()))
        top2 = torch.topk(lg, 2, dim=1).values
        clear = ((top2[:, 0] - top2[:, 1]) / sc > BOUND_LOGIT).cpu().numpy()
        am = torch.argmax(lg, 1).cpu().numpy()
        assert np.array_equal(dec[clear], am[clear]), ("not the float64 argmax at a clear margin", r)
        if len(row0) and row0[0] in idx:
            j = int(np.nonzero(idx == row0[0])[0][0])
            e = float((torch.as_tensor(tap[r].astype(np.float64), device=ref.dev) - lg[j]).abs().max() / sc[j])
            worst["logit"] = max(worst["logit"], e)
        st.apply(idx, dec)
    # final state: counts, prev_token, par and cand_valid exactly; h / c (both parities) and dec_proj against float64
    assert np.array_equal(out["counts"][rows], st.emitted)
    assert np.array_equal(out["prev_token"][slots], st.prev.cpu().numpy())
    assert np.array_equal(out["par"][slots], (par0 + st.emitted) % 2)
    assert np.array_equal(out["cand_valid"][slots], st.valid.cpu().numpy().astype(np.int32))
    parf = out["par"][slots]
    valid = st.valid
    other_h = torch.where(valid[:, None], st.ch, st.old_h)
    other_c = torch.where(valid[:, None], st.cc, st.old_c)
    # a slot that never emitted and never refreshed keeps its input candidate in the other parity (old_* starts there)
    for got, want in ((pick(out["h"], parf), st.h), (pick(out["c"], parf), st.c), (pick(out["h"], 1 - parf), other_h),
                      (pick(out["c"], 1 - parf), other_c), (out["dec_proj"][slots], st.proj)):
        g = torch.as_tensor(got.astype(np.float64), device=ref.dev)
        worst["state"] = max(worst["state"], float(((g - want).abs() / (want.abs() + 1)).max()))
    assert worst["state"] <= BOUND_STATE, worst
    assert worst["logit"] <= BOUND_LOGIT, worst
    return worst


def sample_rows(B, k=48, seed=0):
    if B <= k:
        return np.arange(B)
    return np.unique(np.concatenate([[0, B - 1], np.random.default_rng(seed).choice(B, k - 2, replace=False)]))


def all_launches(eng, ref, inp, rows, case, T, launches=tuple(LAUNCHES)):
    """every launch of `launches` on inp: bit-identical to the first; the first against float64 (identical bits pass the same
    check); row 0 against its own logits -> (first output, decision sequences, templates reached per launch)"""
    first = run(eng, inp, launches[0])
    seqs, per_frame = decisions(first, T)
    check_row0(first, seqs)
    worst = check_f64(ref, inp, first, seqs, rows)
    need, act = round_counts(seqs, inp["cand_valid"][inp["slot_of_b"]])
    reached = {launches[0]: templates(launches[0], need, act)}
    for ln in launches[1:]:
        assert_same(first, run(eng, inp, ln), ln)
        reached[ln] = templates(ln, need, act)
    report(test=case, rows=len(rows), evals=int(sum(len(s) for s in seqs)), tokens=int(first["counts"].sum()),
           templates={k: sorted(v) for k, v in reached.items()}, **worst, bound_logit=BOUND_LOGIT, bound_state=BOUND_STATE)
    return first, seqs, per_frame, reached, (need, act)


# ---- dispatch matrix ---------------------------------------------------------------------------------------------------------
# A quarter of the frames forced towards blank or a token, the rest natural, so the active and emitting counts change from round to
# round. Templates the six launches reach together (the union over the matrix must be all eight, asserted below):
#   B1_T14, B8_T7: phase<1>, pipe<1,1>, gemv<1>            B9_T14, B16_T2: phase<1|2>, pipe<1,1>, <1,2>, gemv<1|2>
#   B17_T7, B65_T7: all eight                               B64_T2: phase<1|2>, pipe<1,1>, <1,4>, <2,4>, gemv<1>
#   B200_T2: phase<2>, pipe<1,2>, <1,4>, <2,4>, gemv<2>     B1024_T1: pipe<2,4> (more than 64 streams in every phase)
MATRIX = [(1, 14), (8, 7), (9, 14), (16, 2), (17, 7), (64, 2), (65, 7), (200, 2), (1024, 1)]
_reached = set()


@pytest.mark.gpu
@pytest.mark.parametrize("B,T", MATRIX, ids=[f"B{b}_T{t}" for b, t in MATRIX])
def test_dispatch_matrix(dec, B, T):
    eng, ref = dec("plain")
    rng = np.random.default_rng(100 + B * 31 + T)
    inp = inputs(ref, B, T, rng, frac_forced=0.25)
    out, seqs, _, reached, _ = all_launches(eng, ref, inp, sample_rows(B), f"matrix_B{B}_T{T}", T)
    assert out["counts"].sum() > 0
    for v in reached.values():
        _reached.update(v)


@pytest.mark.gpu
def test_dispatch_matrix_reaches_every_template(dec):
    """runs after the matrix: together its cases reached all eight device templates"""
    if not _reached:
        pytest.skip("the dispatch matrix did not run in this session")
    assert _reached == ALL_TEMPLATES, ALL_TEMPLATES - _reached


# ---- schedules that cross the dispatch thresholds inside one call ------------------------------------------------------------
@pytest.mark.gpu
def test_schedule_crosses_thresholds(dec):
    """B = 200, T = 4: each stream's leading frames forced to blank, the rest to a token (10 emissions each). A stream with k token
    frames takes 4 + 9 k evaluations; 135 / 48 / 8 / 1 / 8 streams with k = 0 / 1 / 2 / 3 / 4 make the active count
    200 -> 65 -> 17 -> 9 -> 8 and the emitting count 200, 8, 9, 17, 65, 17, 9, 8: both sides of 64 / 65, 16 / 17 and 8 / 9.
    Templates: all eight across the six launches."""
    eng, ref = dec("plain")
    B, T = 200, 4
    ks = np.repeat([0, 1, 2, 3, 4], [135, 48, 8, 1, 8])
    rng = np.random.default_rng(7)
    perm = rng.permutation(B)                                                 # the groups interleaved over the batch rows
    k_of = ks[perm]
    inp = inputs(ref, B, T, rng)
    for b in range(B):
        tok = int(rng.integers(0, BLANK))
        for t in range(T):
            inp["enc_proj"][b, t] = forced(ref, tok if t >= T - k_of[b] else BLANK)
    rows = np.unique(np.concatenate([[0], [np.nonzero(k_of == k)[0][0] for k in range(5)], sample_rows(B, 24, 1)]))
    out, seqs, per_frame, reached, (need, act) = all_launches(eng, ref, inp, rows, "schedule", T)
    assert np.array_equal(out["counts"], 10 * k_of)                          # every forced frame did what it was forced to
    assert np.array_equal(per_frame, np.where(np.arange(T)[None] >= T - k_of[:, None], 10, 0))
    for pat in ((65, 17), (17, 9), (9, 8)):
        assert any(act[i] == pat[0] and act[i + 1] == pat[1] for i in range(len(act) - 1)), (pat, act)
    for lo, hi in ((64, 65), (16, 17), (8, 9)):
        assert any(n <= lo for n in need if n) and any(n >= hi for n in need), (lo, hi, need)
    assert set().union(*reached.values()) == ALL_TEMPLATES, ALL_TEMPLATES - set().union(*reached.values())


# ---- symbol cap ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_symbol_cap(dec):
    """every frame forced towards a token: 10 emissions per frame, the frame advances with no blank evaluation (the tap counts
    exactly 10 T evaluations of row 0), the 10 T output entries are all used and the guards behind them untouched, no candidate
    is left valid. B = 9: phase<2> on the full grid; gemv<2> and pipe<1,2> on 20 CTAs."""
    eng, ref = dec("plain")
    B, T = 9, 7
    rng = np.random.default_rng(11)
    inp = inputs(ref, B, T, rng)
    toks = rng.integers(0, BLANK, B)
    for b in range(B):
        inp["enc_proj"][b, :] = forced(ref, int(toks[b]))
    out, seqs, per_frame, _, _ = all_launches(eng, ref, inp, np.arange(B), "cap", T, launches=("full", "narrow20"))
    assert np.all(out["counts"] == MAX_SYMBOLS * T)
    assert np.all(out["tokens"] == toks[:, None])
    assert np.array_equal(out["frames"], np.repeat(np.arange(T), MAX_SYMBOLS)[None].repeat(B, 0))
    assert out["n_logits"] == MAX_SYMBOLS * T
    assert np.all(out["cand_valid"] == 0) and np.all(out["par"] == (MAX_SYMBOLS * T) % 2)


@pytest.mark.gpu
def test_symbol_cap_batch_path_shape(dec):
    """B = 1, T = 2048 (the batch path's longest utterance), every other frame forced towards a token: 10 240 emissions and
    11 264 evaluations through the kernel's 16-bit counters. phase<1> on the full grid."""
    eng, ref = dec("plain")
    B, T = 1, 2048
    rng = np.random.default_rng(12)
    inp = inputs(ref, B, T, rng)
    toks = rng.integers(0, BLANK, T)
    for t in range(T):
        inp["enc_proj"][0, t] = forced(ref, int(toks[t]) if t % 2 == 0 else BLANK)
    out, seqs, per_frame, _, _ = all_launches(eng, ref, inp, [0], "cap_T2048", T, launches=("full",))
    assert int(out["counts"][0]) == MAX_SYMBOLS * T // 2
    assert np.array_equal(per_frame[0], np.where(np.arange(T) % 2 == 0, MAX_SYMBOLS, 0))
    assert np.array_equal(out["tokens"][0, :MAX_SYMBOLS * T // 2], np.repeat(toks[::2], MAX_SYMBOLS))
    assert out["n_logits"] == MAX_SYMBOLS * T // 2 + T // 2


# ---- exact ties ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("rot", [0, 1, 2])
def test_exact_ties(dec, rot):
    """the tie model (_tie_model): 8 streams forced towards 16 (tied with 17 in one item / tile), 8 towards 3 (tied with 1000 in
    another CTA), 8 towards blank (tied with 500); batch row 0 is one of each group in turn. The tapped logits of each pair are
    bitwise equal (precondition); the lower index wins on every launch, a token tied with blank emits. B = 24, T = 2: phase<2>,
    pipe<1,4>, pipe<2,4>."""
    eng, ref = dec("tie")
    B, T = 24, 2
    rng = np.random.default_rng(20)
    inp = inputs(ref, B, T, rng)
    target = np.roll(np.repeat([16, 3, BLANK], 8), -8 * rot)
    for b in range(B):
        inp["enc_proj"][b, :] = forced(ref, int(target[b]))
    out, seqs, _, _, _ = all_launches(eng, ref, inp, np.arange(B), f"ties_rot{rot}", T)
    lg = out["logits"]
    for hi, lo in TIE_PAIRS:
        assert np.array_equal(lg[:, hi].view(np.uint32), lg[:, lo].view(np.uint32)), (hi, lo)
    winner = {16: 16, 3: 3, BLANK: 500}
    assert np.all(out["counts"] == MAX_SYMBOLS * T)
    for b in range(B):
        assert np.all(out["tokens"][b] == winner[int(target[b])]), (b, target[b], out["tokens"][b][:4])


# ---- row 0 against its own logits, rotated ------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("shift", [0, 5, 11])
def test_row0_logits_rotated(dec, shift):
    """the same 17 streams with a different stream as batch row 0: its token at every evaluation is the first argmax of its own
    tapped logits, those logits match float64, and every stream decodes the same whatever its row. B = 17, T = 7 on 20 CTAs
    (gemv<1|2>, pipe<1,1>, <1,2>, <1,4>, <2,4>) and the full grid (phase<1|2>)."""
    eng, ref = dec("plain")
    B, T = 17, 7
    base = inputs(ref, B, T, np.random.default_rng(30), frac_forced=0.25)
    inp = dict(base, enc_proj=np.roll(base["enc_proj"], -shift, axis=0))
    out, _, _, _, _ = all_launches(eng, ref, inp, np.arange(B), f"row0_shift{shift}", T, launches=("narrow20", "full"))
    ref_out = run(eng, base, "full")
    back = lambda a: np.roll(a, shift, axis=0)
    for k in ("tokens", "frames", "counts"):
        assert np.array_equal(back(out[k]), ref_out[k]), k


# ---- carried state ------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("B,S", [(40, 100), (130, 300)], ids=["B40_S100", "B130_S300"])
def test_carried_state(dec, B, S):
    """state a step leaves behind: random committed h / c at parity 0 or 1, non-blank prev_token, and on half the slots a valid
    candidate whose dec_proj is deliberately NOT its projection (the kernel must use it until the first emission); the batch
    decodes a random subset of S slots in random order. Slots outside the batch come back bit for bit unchanged.
    B = 40: phase<1|2>, gemv<1|2> and pipe<1,1> .. <2,4>; B = 130 adds pipe<2,4> on the wide grids."""
    eng, ref = dec("plain")
    T = 3
    rng = np.random.default_rng(40 + B)
    inp = inputs(ref, B, T, rng, S=S, frac_forced=0.2)
    inp["slot_of_b"] = rng.choice(S, B, replace=False).astype(np.int32)
    inp["h"] = np.tanh(rng.standard_normal((S, 2, 2 * HID))).astype(np.float32)
    inp["c"] = rng.standard_normal((S, 2, 2 * HID)).astype(np.float32)
    inp["dec_proj"] = rng.standard_normal((S, HID)).astype(np.float32)
    inp["par"] = rng.integers(0, 2, S).astype(np.int32)
    inp["prev_token"] = rng.integers(0, BLANK, S).astype(np.int32)
    inp["cand_valid"] = rng.integers(0, 2, S).astype(np.int32)
    rows = sample_rows(B)
    out, seqs, _, _, _ = all_launches(eng, ref, inp, rows, f"carried_B{B}_S{S}", T,
                                      launches=("full", "narrow20", "full_pipe1", "plain96"))
    # the carried candidate was used: a stream with a valid candidate decides its first evaluation on the given dec_proj
    assert any(inp["cand_valid"][inp["slot_of_b"][b]] and seqs[b][0][1] != BLANK for b in range(B))
    outside = np.setdiff1d(np.arange(S), inp["slot_of_b"])
    for k in ("h", "c", "dec_proj", "par", "prev_token", "cand_valid"):
        assert np.array_equal(np.asarray(out[k])[outside].view(np.uint32), np.asarray(inp[k])[outside].view(np.uint32)), k


# ---- argument errors ----------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_argument_errors_write_nothing(dec):
    """every rejected argument returns NSB_ERR_ARG and leaves every output array and field as it was"""
    import nsb200
    eng, ref = dec("plain")
    L = nsb200.lib()
    B, T, S = 4, 2, 6
    rng = np.random.default_rng(50)
    good = inputs(ref, B, T, rng, S=S)
    good["slot_of_b"] = np.array([5, 0, 3, 1], np.int32)
    sms = sm_count()

    def call(B=B, T=T, S=S, grid=0, pipe=0, null_enc=False, **over):
        a = {k: np.ascontiguousarray(v).copy() for k, v in good.items()}
        a.update({k: np.ascontiguousarray(v) for k, v in over.items()})
        outs = dict(tokens=np.full(max(B, 1) * 10 * max(T, 1), 77, np.int32), frames=np.full(max(B, 1) * 10 * max(T, 1), 77, np.int32),
                    counts=np.full(max(B, 1), 77, np.int32), logits=np.full(16, 7.0, np.float32))
        before = {k: v.copy() for k, v in list(a.items()) + list(outs.items())}
        p = lambda x: x.ctypes.data_as(C.c_void_p)
        op = nsb200.DecodeOp(B, T, S, grid, pipe, p(a["slot_of_b"]), None if null_enc else p(a["enc_proj"]), p(a["h"]), p(a["c"]),
                             p(a["dec_proj"]), p(a["par"]), p(a["prev_token"]), p(a["cand_valid"]), p(outs["tokens"]),
                             p(outs["frames"]), p(outs["counts"]), p(outs["logits"]), 123, 456, 789)
        rc = L.nsb_op_decode(eng.h, C.byref(op))
        msg = L.nsb_last_error().decode()
        assert rc == -1, (rc, msg)
        for k, v in before.items():
            now = a.get(k, outs.get(k))
            assert np.array_equal(now.view(np.uint8), v.view(np.uint8)), f"{k} written by a rejected call ({msg})"
        assert (op.n_logits, op.grid_used, op.guard_bad) == (123, 456, 789)
        return msg

    big = lambda n: dict(slot_of_b=np.arange(n, dtype=np.int32), **{k: np.resize(v, (n,) + v.shape[1:]) for k, v in good.items()
                                                                      if k not in ("slot_of_b", "enc_proj")},
                         enc_proj=np.resize(good["enc_proj"], (n, T, HID)))
    assert "B must" in call(B=0)
    assert "B must" in call(B=1025, S=1025, **big(1025))
    assert "T must" in call(T=0)
    assert "T must" in call(T=3277, enc_proj=np.zeros((B, 3277, HID), np.float32))
    assert "S must" in call(S=3)
    assert "S must" in call(S=8193)
    assert "slot_of_b" in call(slot_of_b=np.array([5, 0, 3, 6], np.int32))
    assert "slot_of_b" in call(slot_of_b=np.array([5, 0, -1, 1], np.int32))
    assert "slot_of_b" in call(slot_of_b=np.array([5, 0, 5, 1], np.int32))
    for v in (-1, 1025):
        assert "prev_token" in call(prev_token=np.where(np.arange(S) == 2, v, BLANK).astype(np.int32))
    for v in (-1, 2):
        assert "par must" in call(par=np.where(np.arange(S) == 4, v, 0).astype(np.int32))
        assert "cand_valid" in call(cand_valid=np.where(np.arange(S) == 4, v, 0).astype(np.int32))
    for g in (-2, 1, 3, 21, sms, sms + 2):
        assert "grid" in call(grid=g)
    assert "pipe_min_n" in call(pipe=-1)
    assert "null" in call(null_enc=True)
