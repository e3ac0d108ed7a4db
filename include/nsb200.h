/* nsb200.h -- C ABI of the B200-native streaming ASR engine (libnsb200.so).
 *
 * This is the drop-in boundary for the ONE hot path of m1el/nemotron-speech.cpp:
 *   16 kHz s16le PCM -> log-mel -> dw-striding subsampling -> N cache-aware FastConformer
 *   layers -> RNN-T (LSTM prediction net + joint) greedy decode, for many independent streams.
 *
 * Plain C, opaque handles, int status (0 = ok, <0 = error; text via nsb_last_error()).
 * No torch / ggml / C++ types cross this boundary. Every entry point cites the reference
 * interface it replaces (paths relative to the reference repo).
 *
 * There is NO CPU fallback: every call that computes runs hand-written sm_100a kernels and
 * fails with NSB_ERR_CUDA when no CUDA device is usable.
 */
#ifndef NSB200_H
#define NSB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NSB_OK 0
#define NSB_ERR_ARG (-1)
#define NSB_ERR_IO (-2)
#define NSB_ERR_FORMAT (-3)
#define NSB_ERR_CUDA (-4)
#define NSB_ERR_STATE (-5)
#define NSB_ERR_NOMEM (-6)

/* arithmetic the per-layer weight GEMMs run in (what ggml picks from the tensor type,
 * src/nemo-ggml.cpp:187-191 "quantized tensors stay quantized, ggml_mul_mat handles dequant") */
enum nsb_compute {
    NSB_COMPUTE_AUTO = 0, /* from the GGUF tensor type: F32 -> F32, F16 -> F16, Q8_0 / Q4_0 -> quantised in HBM, fp16 tensor-core GEMMs */
    NSB_COMPUTE_F32 = 1,  /* SIMT fp32 GEMM (strict parity with the f32 reference path)                   */
    NSB_COMPUTE_F16 = 2,  /* tcgen05 kind::f16, fp16 operands, fp32 TMEM accumulate                       */
    NSB_COMPUTE_BF16 = 3, /* tcgen05 kind::f16, bf16 operands, fp32 TMEM accumulate                       */
    NSB_COMPUTE_Q8_0 = 4, /* Q8_0 weights resident in HBM, dequantised to fp16 in the operand producer    */
    NSB_COMPUTE_Q8_0_STRICT = 5 /* the reference's own Q8_0 arithmetic (ggml_mul_mat on a Q8_0 src0): activation rows quantised
                                   per 32 (d = amax/127 as fp16, q = roundf(x/d)), exact integer block dots on the tensor cores
                                   (mma s8), f32 scale-accumulate in block order; everything else as NSB_COMPUTE_F32. Parity mode */
};
enum nsb_kv_dtype { NSB_KV_F32 = 0, NSB_KV_F16 = 1, NSB_KV_BF16 = 2 };

typedef struct nsb_engine nsb_engine;

typedef struct nsb_engine_config {
    int32_t device;            /* CUDA ordinal                                                         */
    int32_t compute;           /* enum nsb_compute                                                     */
    int32_t kv_dtype;          /* enum nsb_kv_dtype: storage of the per-stream K/V ring                */
    int32_t att_right_context; /* R in {0,1,6,13}: nemo_cache_config::att_right_context (nemo-stream.h:26) */
    int32_t max_streams;       /* stream slots resident on this GPU                                    */
    int32_t use_cuda_graph;    /* capture the per-step launch sequence per batch size                  */
    int32_t decode_overlap;    /* RNN-T decode of step i on its own stream, on a few SMs, under the encoder of step i+1:
                                  0 = automatic (steps of <= 512 token rows that are begun while another step is in flight),
                                  1 = always, 2 = never. Same tokens either way */
    int32_t reserved[5];
} nsb_engine_config;

typedef struct nsb_stats {
    int64_t steps;             /* engine steps run                                                     */
    int64_t chunks;            /* stream-chunks processed (sum over streams)                           */
    int64_t kernel_launches;   /* kernels of this library launched                                     */
    double device_ms;          /* CUDA-event time of all steps                                         */
    double last_step_ms;
} nsb_stats;

/* ---- GGUF metadata without touching the GPU: what nemo_model_load reads before the tensor data
 *      (src/nemo-ggml.cpp:99-146: nemo.* hparams and tokenizer.vocab) ------------------------ */
typedef struct nsb_model_info {
    int32_t n_mels, d_model, n_heads, d_head, d_ff, n_layers, kernel_size, vocab_size, decoder_dim, joint_dim;
    int32_t n_tensors;
    int32_t weight_type;      /* ggml type of the per-layer matrices: 0 F32, 1 F16, 2 Q4_0, 8 Q8_0 */
    char vocab[1025 * 8];     /* char8 pieces, NUL padded (bounded copy + zero fill)        */
} nsb_model_info;
int nsb_gguf_probe(const char* gguf_path, nsb_model_info* info);
/* One tensor of the file as floats, as the engine's loader sees it (F32 / F16 as stored, Q8_0 / Q4_0 dequantised like ggml's
 * dequantize_row_*; scripts/convert_to_gguf.py:93-179), also without a GPU. Returns the element count (out == NULL: query only), or
 * <0 with nsb_last_error() (missing tensor, unsupported type, buffer too small); *ggml_type (optional) = the stored type. */
long long nsb_gguf_read_tensor(const char* gguf_path, const char* tensor_name, float* out, size_t cap_floats, int* ggml_type);

/* ---- engine lifetime: replaces nemo_init_with_backend / nemo_model_load / nemo_free
 *      (src/nemo-ggml.h:231-242, src/nemo-ggml.cpp:83-463) --------------------------------- */
void nsb_default_config(nsb_engine_config* cfg);
int nsb_engine_create(const char* gguf_path, const nsb_engine_config* cfg, nsb_engine** out);
void nsb_engine_destroy(nsb_engine* e);
const char* nsb_last_error(void);

/* model facts (src/nemo-ggml.h:37-49 nemo_hparams; :157-160 char8 vocab) */
int nsb_engine_n_layers(const nsb_engine* e);
int nsb_engine_vocab_size(const nsb_engine* e);
const char* nsb_engine_vocab(const nsb_engine* e); /* vocab_size * 8 bytes, NUL padded */
int nsb_engine_chunk_samples(const nsb_engine* e); /* nemo_cache_config::get_chunk_samples (nemo-stream.h:85-87) */
int nsb_engine_shift_samples(const nsb_engine* e); /* 160 * get_shift_mel_frames (nemo-stream.h:76-81)          */
int nsb_engine_compute(const nsb_engine* e);       /* resolved enum nsb_compute                                  */
/* switch CUDA-graph replay of the step on / off at run time (nsb_engine_config::use_cuda_graph is the initial value). Both ways
 * launch the same kernels with the same arguments: results are bit-identical (bench.py checks a token checksum across the two). */
int nsb_engine_set_cuda_graph(nsb_engine* e, int on);

/* ---- streams: replaces nemo_stream_init / reset / free (src/nemo-stream.h:262-312) ------- */
int nsb_stream_open(nsb_engine* e);                /* returns stream id >= 0, or <0 */
int nsb_stream_close(nsb_engine* e, int stream);
int nsb_stream_reset(nsb_engine* e, int stream);   /* re-zeroes caches too (the reference's reset does not) */

/* ---- stream snapshots: suspend, resume and move live streams (no counterpart in the reference) --------------------------
 * A snapshot holds everything that decides the stream's future output: its K/V ring, conv state, mel overlap and decoder state,
 * the PCM buffered for chunks not yet launched, its chunk counters and the tokens not yet popped. Engine statistics are not part
 * of it. Callers treat it as opaque bytes (layout: DESIGN.md §11). Both calls collect the steps in flight first, like open / close.
 * nsb_stream_export: the stream stays open and continues exactly as if nothing happened (tokens of the steps that were in flight
 *   are in the snapshot and stay poppable on the stream). out == NULL: returns the size an export would write now. Returns the
 *   bytes written; a closed stream, an invalid id, or cap smaller than the size is NSB_ERR_ARG (the buffer is left untouched).
 *   Suspend = export, then close; move = export on A, import on B, close on A.
 * nsb_stream_import: takes the lowest free slot like nsb_stream_open and returns the new stream id. The engine must run the same
 *   model (a fingerprint of the GGUF: metadata, tensor table, first and last 4 KiB of every tensor -- the path does not matter),
 *   n_layers, att_right_context, kv_dtype and resolved compute; device, max_streams, use_cuda_graph and decode_overlap may differ.
 *   NSB_ERR_FORMAT: not a valid snapshot (magic, version, size, checksum, a field out of range); NSB_ERR_ARG: a valid snapshot that
 *   does not fit this engine; NSB_ERR_STATE: no free slot. nsb_last_error() names the field. A failed import changes nothing:
 *   no slot is consumed and no other stream is touched. */
long long nsb_stream_export(nsb_engine* e, int stream, void* out, size_t cap);
int nsb_stream_import(nsb_engine* e, const void* snapshot, size_t bytes);

/* ---- the hot call: replaces nemo_stream_process_incremental (src/nemo-stream.cpp:1074-1134)
 *      split into push (buffer PCM, any length) / step (one batched chunk for every stream that
 *      has a full chunk buffered) / pop (token ids decoded so far). ------------------------- */
int nsb_stream_push_pcm(nsb_engine* e, int stream, const int16_t* pcm, int n_samples);
/* the same for many streams in one call (a serving loop feeds every stream once per chunk period): row i of `pcm`
 * (row_stride samples apart) goes to streams[i]; tokens of streams[i] land in out[i * cap_per_stream ..], counts[i] = how many.
 * pop returns the total number of tokens copied. */
int nsb_push_pcm_batch(nsb_engine* e, int n_streams, const int32_t* streams, const int16_t* pcm, int row_stride, int n_samples);
int nsb_pop_tokens_batch(nsb_engine* e, int n_streams, const int32_t* streams, int32_t* out, int cap_per_stream, int32_t* counts);
int nsb_stream_ready(const nsb_engine* e, int stream); /* 1 if a full chunk is buffered */
int nsb_engine_step(nsb_engine* e);                    /* returns #streams advanced (0 = nothing ready), <0 error */
/* step() split in two so that the host can feed the NEXT chunk while the device works on this one: begin stages the ready
 * streams, enqueues the H2D copy, the step and the D2H copy of the token ids and returns; end waits for them and queues the
 * tokens of the OLDEST step in flight. Up to three steps may be in flight (begin, begin, [begin,] end, begin, end, ...: the device
 * goes from one step straight into the next; with a third step queued the engine stream also stays busy while the greedy decode of a
 * step with many symbols is still running on its own stream; a fourth begin is an error); push_pcm / pop_tokens are allowed in between, stream open / close /
 * reset and nsb_engine_step collect first. nsb_stream_ready() counts launched chunks (it asks for the chunk after the ones in
 * flight); nsb_stream_chunks() counts collected ones. */
int nsb_engine_step_begin(nsb_engine* e);              /* returns #streams in the launched step (0 = nothing ready), <0 error */
int nsb_engine_step_end(nsb_engine* e);                /* returns #streams advanced (0 = no step in flight), <0 error */
int nsb_engine_drain(nsb_engine* e);                   /* step until nothing is ready; returns total stream-chunks */
int nsb_stream_pop_tokens(nsb_engine* e, int stream, int32_t* out, int cap); /* returns n copied (FIFO) */
int nsb_stream_chunks(const nsb_engine* e, int stream);                      /* nemo_stream_context::total_chunks_processed */

/* tokens_to_text (src/nemo-ggml.cpp:1432-1458, no timestamps). Returns bytes written (excl. NUL) or -needed */
int nsb_detokenize(const nsb_engine* e, const int32_t* tokens, int n, char* out, int cap);

void nsb_engine_get_stats(const nsb_engine* e, nsb_stats* out);

/* ---- benchmarking hooks (device-resident inputs; no PCIe inside the timed region) --------
 * nsb_bench_prepare: open `n_streams` streams, warm their caches by running `warm_chunks` chunks
 * of synthetic audio, and stage every further full chunk of PCM the caller supplied (at least one, at most 16) in HBM.
 * nsb_bench_step: run ONE batched step over all those streams from the staged PCM, cycling through the staged chunks
 * (state advances; tokens are produced and discarded). Returns device ms of the step via *ms. */
int nsb_bench_prepare(nsb_engine* e, int n_streams, const int16_t* pcm, int samples_per_stream, int warm_chunks);
int nsb_bench_step(nsb_engine* e, float* ms);
/* n steps enqueued back to back (no host synchronisation in between), one CUDA event between consecutive steps:
 * ms_each[i] (optional, n floats) = device time of step i, *total_ms = first event -> last event */
int nsb_bench_steps(nsb_engine* e, int n, float* ms_each, float* total_ms);
/* one bench step with every kernel launch bracketed by CUDA events on the engine's stream; device ms and launch
 * count per kernel class: 0 log-mel, 1 subsampling, 2 layernorm, 3 layer GEMMs, 4 attention, 5 conv module,
 * 6 joint.enc + RNN-T decode, 7 misc. Arrays must hold NSB_PROFILE_CLASSES entries. */
#define NSB_PROFILE_CLASSES 8
int nsb_bench_profile(nsb_engine* e, float* ms_per_class, int* launches_per_class, float* total_ms);

/* tuning hook: `iters` passes over every layer's weight of one kind (0 ff1.linear1, 1 ff1.linear2, 2 qkv, 3 attn out, 4 pw1,
 * 5 pw2) with an explicit tcgen05 tile config (bn, stages, split-K, k rotation); *us = mean device microseconds per GEMM */
int nsb_bench_gemm(nsb_engine* e, int kind, int rows, int bn, int stages, int splits, int rotate, int iters, float* us);

/* ---- in-situ device trace: block 0 of every kernel stamps %globaltimer (ns) at start [0], after it stopped waiting for the
 * previous kernel [1] (GEMM: prologue done [1], wait returned [2], accumulator complete [3], epilogue done [4]) and at its end [2].
 * Works inside the CUDA graph, where ncu cannot look. tag: 1 log-mel, 2 stem, 3 dwconv, 4 mel history, 5 fp32 GEMM, 6 tcgen05 GEMM,
 * 7 Q8_0 GEMM, 8 LayerNorm, 9 fused double LayerNorm, 10 attention, 11 conv module, 12 advance, 13 decode. capacity 0 = off. */
typedef struct nsb_trace_record { uint64_t t[6]; int32_t tag; int32_t grid; } nsb_trace_record;
int nsb_trace_enable(nsb_engine* e, int capacity);
int nsb_trace_fetch(nsb_engine* e, nsb_trace_record* out, int cap); /* returns #records copied, resets the trace */

/* cudaProfilerStart / cudaProfilerStop, so that `ncu --profile-from-start off` captures only the steady-state steps */
int nsb_profiler_range(int on);

/* ---- parity / debug taps (host buffers) --------------------------------------------------
 * When enabled, the engine keeps the tensors of the LAST step: names
 *   "mel" [B, M, 128]  "sub" [B*T, 1024]  "layer.<l>" [B*T, 1024]  "enc" [B*T, 1024]
 * and, for decode, every joint evaluation's logits of batch row 0 ("logits", up to cap evals).
 * Rows are ordered by the step's batch order = ascending stream id.
 * One name works WITHOUT tap mode: "x" [B*T, 1024] = encoder output of the most recently launched step, copied out of the step
 * workspace after the step -- it observes the production path (CUDA graph, no taps) unchanged. */
int nsb_debug_enable(nsb_engine* e, int on);
int nsb_debug_get(nsb_engine* e, const char* name, float* out, size_t cap_floats); /* returns #floats or <0 */
int nsb_debug_get_cache(nsb_engine* e, int stream, int which /*0=k,1=v,2=conv*/, int layer, float* out, size_t cap);

/* ---- stand-alone operators (unit parity against the oracle; host in / host out) ----------
 * nsb_op_logmel: nemo_preprocessor_process (src/preprocessor.cpp:330-395) for a batch of
 *   independent streams starting at stream start: pcm [n_streams, n_samples] -> mel
 *   [n_streams, n_frames, 128]; returns n_frames = (256 + n_samples - 512)/160 + 1.
 * nsb_op_gemm: y[rows, n_out] = x[rows, n_in] * W^T for a named per-layer weight, in the
 *   engine's compute arithmetic (ggml_mul_mat, e.g. src/nemo-stream.cpp:571-573). */
int nsb_op_logmel(nsb_engine* e, const int16_t* pcm, int n_streams, int n_samples, float* mel_out, size_t cap_floats);
int nsb_op_gemm(nsb_engine* e, const char* weight_name, const float* x, int rows, float* y, size_t cap_floats);

/* ---- operator tests of the step's GEMM and LayerNorm launches (host in / host out) ----------------------------------------
 * nsb_op_gemm_ex: one GEMM C = epi(x W^T) on a weight nsb_op_gemm takes (per-layer matrices, and the matrices every GGUF keeps in
 *   F32: encoder.pre_encode.conv.3 / conv.6 / out, joint.enc -- 3xTF32 on the tensor cores; pre_encode.out expects x in the engine's
 *   (w * 256 + c) column order), launched through the engine's own dispatch with the settings below. x [rows][n_in] f32 is rounded to
 *   the engine's activation type like the step's producers (F32 matrices: plain f32). The destination (and the split-K workspace) is
 *   padded with guard rows before and after the live region and 32 unused columns per row (ldc = n_out + 32), all holding a NaN
 *   pattern; *guard_bad = how many guard elements the GEMM changed (0 = no stray store).
 *   y receives the raw output bits: [m_out][n_out] elements of out_type (16-bit outputs as stored, 2 bytes each), or for
 *   NSB_EPI_PARTIAL every k-slice plane [splits][m_out][n_out] f32 (plane 0 from C0 when c0 is set). m_out = rows, or with the
 *   output row map rows / c_group * (c_group - c_drop). Returns n_out, -bytes needed when y_bytes is too small, <0 on error (a forced
 *   tile config that is not instantiated for the operand type or whose grid does not cover n_out is NSB_ERR_ARG). */
enum nsb_epi { NSB_EPI_NONE = 0, NSB_EPI_RELU = 1, NSB_EPI_SILU = 2, NSB_EPI_RESID = 3, NSB_EPI_PARTIAL = 4 };
enum nsb_out_type { NSB_OUT_F32 = 0, NSB_OUT_F16 = 1, NSB_OUT_BF16 = 2 };
typedef struct nsb_gemm_op {
    const char* weight;        /* tensor name                                                                             */
    int32_t rows;              /* rows of x (M)                                                                           */
    int32_t epi;               /* enum nsb_epi: NONE / RELU (+bias) / SILU / RESID (C += alpha acc, f32) / PARTIAL (split-K)  */
    float alpha;               /* NSB_EPI_RESID                                                                           */
    int32_t out_type;          /* enum nsb_out_type; 16-bit only for NONE / RELU / SILU                                   */
    int32_t splits;            /* k slices (NSB_EPI_PARTIAL; 1 otherwise)                                                 */
    int32_t c0;                /* NSB_EPI_PARTIAL: slice 0 (+ bias) goes to its own destination, slices z >= 1 to workspace plane z-1 */
    int32_t c_group, c_drop;   /* output row map: rows r with r % c_group < c_drop are dropped, the rest compacted (0 = off)  */
    int32_t force_bn, force_stages;   /* tile config as nsb_bench_gemm takes it; 0 = the engine's own dispatch             */
    int32_t rotate;            /* CTA n starts its k loop at k-block (n mod nk) (single-CTA tiles)                        */
    const float* bias;         /* [n_out] or NULL                                                                         */
    const float* c_init;       /* NSB_EPI_RESID: initial C [m_out][n_out]                                                 */
} nsb_gemm_op;
int nsb_op_gemm_ex(nsb_engine* e, const nsb_gemm_op* op, const float* x, void* y, size_t y_bytes, long long* guard_bad);
/* nsb_op_decode: the step's RNN-T greedy-decode launch (LSTM prediction net, joint.pred, joint, argmax, up to 10 symbols per frame)
 *   on the engine's decoder weights, for B streams of T frames each. enc_proj [B][T][640] f32 is what joint.enc produced (bias
 *   included). The decoder state of S >= B slots comes in and goes out in the engine's layout: h, c [S][2 parities][2 layers x 640]
 *   (committed state at parity par[s], candidate at the other), dec_proj [S][640] (joint.pred projection of the candidate), par,
 *   prev_token (0..1024), cand_valid (0 / 1) [S]; batch row b decodes slot slot_of_b[b] (distinct). Device state, sync buffer and
 *   outputs are private to the call: no stream slot is touched. grid = 0: one CTA per SM (cooperative launch, as in a step);
 *   grid = k (even, 2 <= k < SM count): the decode-overlap launch with k CTAs in pairs. pipe_min_n: streams per phase from which
 *   the pipelined tiles run on a wide grid (0 = the engine's default). Outputs: tokens / frames [B][10 T] (entries past counts[b]
 *   keep -1), counts [B], optionally the logits of batch row 0 at each of its joint evaluations, logits [11 T][1025] (*n_logits =
 *   evaluations), the grid used and the number of guard entries behind the token / frame buffers the launch changed. Runs on the
 *   engine stream and synchronises. Returns 0, NSB_ERR_ARG for a bad argument (nothing is written then). */
typedef struct nsb_decode_op {
    int32_t B, T, S;           /* 1 <= B <= 1024, 1 <= T <= 3276 (10 T emissions fit the kernel's 16-bit counters), B <= S <= 8192 */
    int32_t grid, pipe_min_n;  /* launch choice (above)                                                                        */
    const int32_t* slot_of_b;  /* [B]                                                                                          */
    const float* enc_proj;     /* [B][T][640]                                                                                  */
    float* h; float* c;        /* in / out [S][2][1280]                                                                        */
    float* dec_proj;           /* in / out [S][640]                                                                            */
    int32_t* par; int32_t* prev_token; int32_t* cand_valid;   /* in / out [S]                                                 */
    int32_t* tokens; int32_t* frames;   /* out [B][10 T]                                                                       */
    int32_t* counts;           /* out [B]                                                                                      */
    float* logits;             /* out [11 T][1025] or NULL                                                                     */
    int32_t n_logits, grid_used;        /* out                                                                                 */
    long long guard_bad;       /* out                                                                                          */
} nsb_decode_op;
int nsb_op_decode(nsb_engine* e, nsb_decode_op* op);
/* nsb_op_layernorm: the LayerNorm launch of the step on host rows of 1024: x [rows][1024] f32 += alpha * (sum of n_planes split-K
 *   planes [n_planes][rows][1024], 0 <= n_planes <= 8, summed in plane order), then fused = 0: y = LN(x; g1, b1) (x keeps the reduced
 *   rows); fused = 1 (norm_out fused with the next layer's first norm): x = LN(x; g1, b1) and, when g2 is set, y = LN(x; g2, b2).
 *   eps 1e-5. y: [rows][1024] of out_type; x_out: x after the launch. Returns 0 or <0. */
int nsb_op_layernorm(nsb_engine* e, const float* x, int rows, const float* planes, int n_planes, float alpha, const float* g1, const float* b1,
                     const float* g2, const float* b2, int fused, int out_type, float* x_out, void* y);

/* ---- non-streaming batch path: replaces nemo_encode_audio / nemo_transcribe_audio (src/nemo-ggml.cpp:1467-1600) for ONE
 * utterance: whole-utterance log-mel -> subsampling with no carried / dropped frames -> non-cached conformer layers with
 * full-context rel-pos attention -> greedy decode from a fresh decoder state. Validated on hardware against the CPU checker and the
 * fixture generated by the reference's compiled modules (tests/test_zz_batch_path.py). Borrows one free stream slot (decoder / conv
 * state); its activations live in a workspace of their own that grows to the longest utterance seen, so any engine -- whatever
 * max_streams -- takes up to 2048 encoder frames (the reference's positional table, nemo-ggml.cpp:196; about 164 s of audio).
 * Returns the number of tokens decoded (min(n, cap) are copied), <0 on error; token_frames (optional, cap entries) = encoder frame of
 * each token = timed_token::frame_idx (nemo-ggml.cpp:1240; seconds = frame * 1280 / 16000); *n_frames = encoder frames; enc_out
 * (optional) receives [n_frames][1024] floats (returns -needed when enc_cap_floats is too small). */
int nsb_transcribe_full(nsb_engine* e, const int16_t* pcm, int n_samples, int32_t* tokens, int32_t* token_frames, int cap, int* n_frames,
                        float* enc_out, size_t enc_cap_floats);

#ifdef __cplusplus
}
#endif
#endif /* NSB200_H */
