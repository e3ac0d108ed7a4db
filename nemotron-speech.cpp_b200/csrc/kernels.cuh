// kernels.cuh -- launchers of the hand-written sm_100a kernels (internal)
#pragma once
#include "common.cuh"

namespace nsb {

// device tracing: every translation unit with kernels binds the trace buffer into its constant memory (common.cuh)
void trace_bind_frontend(TraceBuf*); void trace_bind_layer(TraceBuf*); void trace_bind_simt(TraceBuf*);
void trace_bind_gemm_tc(TraceBuf*); void trace_bind_decode(TraceBuf*);

// ---------------------------------------------------------------- front-end (kernels_frontend.cu)
// log-mel of n_frames frames per row. Row b of `pcm` holds [prev_sample, s_0, s_1, ...] of the
// 256-zero-left-padded stream; frame j covers s[160 j .. 160 j + 512). Output row stride given.
void launch_logmel(const int16_t* pcm, int pcm_row_stride, int B, int n_frames, const float* window512,
                   const float* cos_t, const float* sin_t, const float* fb_t /*[257][128]*/, float* mel_out,
                   size_t out_batch_stride, cudaStream_t st);

// conv0 (1->256, 3x3 s2, pad 2/1) + ReLU on the chunk image [M = 9 + 8T frames, 128 mels]; frames 0..8 come
// from the per-slot history, the rest from mel_new. Output NHWC [B][t1][65][256].
void launch_conv0(const float* mel_hist, const float* mel_new, const int* slot_of_b, int B, int T, const float* w_t /*[9][256]*/,
                  const float* bias, float* out, cudaStream_t st);
// conv0 + ReLU fused into the first depthwise conv: mel chunk -> [B][t2][33][256] (the conv0 image never reaches HBM)
void launch_stem_conv0_dw(const float* mel_hist, const float* mel_new, const int* slot_of_b, int B, int T, const float* w0_t,
                          const float* b0, const float* w2_t, const float* b2, float* out, cudaStream_t st, int split = 0);
// the same on a whole mel image [B][M][128] of any length M (non-streaming batch path): -> [B][t2][33][256], t2 = (M/2+1)/2+1
void launch_stem_conv0_dw_full(const float* mel, int B, int M, const float* w0_t, const float* b0, const float* w2_t, const float* b2,
                               float* out, cudaStream_t st, int split = 0);
// history = last 9 frames of [hist || new]
void launch_mel_hist_update(float* mel_hist, const float* mel_new, const int* slot_of_b, int B, int T, cudaStream_t st);
// optional tap: full chunk image [B][M][128]
void launch_mel_gather(const float* mel_hist, const float* mel_new, const int* slot_of_b, int B, int T, float* out, cudaStream_t st);
// depthwise 3x3 s2 (+bias), NHWC, C = 256. split = 1 (also launch_stem_conv0_dw): every output pixel is written as 512 floats
// [tf32 hi (256) | tf32 lo (256)] -- the A operand layout of the 3xTF32 tensor-core GEMM that follows (GemmArgs::a_fold)
void launch_dwconv_s2(const float* in, int B, int H, int W, const float* w_t /*[9][256]*/, const float* bias, float* out,
                      cudaStream_t st, int split = 0);
// rows x K fp32 -> rows x [hi (K) | lo (K)]: v = hi + lo (+ <= 2^-22 |v|), both exactly representable in tf32
void launch_split_tf32(const float* in, float* out, size_t rows, int K, cudaStream_t st);

// ---------------------------------------------------------------- SIMT fp32 GEMM (gemm_simt.cu)
struct GemmArgs {
    const void* A = nullptr;      // [M, K] row-major (K contiguous); f32 for SIMT, f16/bf16 for tensor-core
    long long lda = 0;            // elements
    // optional row map: A row(m) = (m / group) * group_stride + (m % group + row_off) * lda   (group == 0 -> m * lda)
    int group = 0; long long group_stride = 0; int row_off = 0;
    const void* W = nullptr;      // [N, K] row-major (Q8_0: the int8 quant plane)
    const void* w_scales = nullptr;   // Q8_0 / Q4_0 only: fp16 block scales [N][K/32]; selects the fused-dequant tensor-core kernel
    int q4 = 0;                       // W is a Q4_0 nibble plane [N][K/2] (two values per byte as in the GGUF block) instead of an int8 plane
    int M = 0, N = 0, K = 0;
    const float* bias = nullptr;  // [N] or null
    void* C = nullptr; long long ldc = 0;
    int epi = EPI_NONE; float alpha = 1.0f; int out_type = OUT_F32;
    int splits = 1;               // split-K factor (EPI_PARTIAL only): C is a [splits][M][N] f32 workspace
    // tensor-core kernel only: output row map (rows r with r % c_group < c_drop are not stored, the rest are compacted) and, for
    // EPI_PARTIAL, an optional destination C0 for k-slice 0 (+bias); slices z >= 1 then go to C[z-1]
    int c_group = 0, c_drop = 0; void* C0 = nullptr;
    int force_bn = 0, force_stages = 0;   // tuning hooks (bench_gemm): pick the tile config explicitly (stages 98 = CTA-pair tile)
    int pair = 0;                 // allow the CTA-pair (cta_group::2) tile when the batch is a single 128-row tile
    int w_dynamic = 0;            // W was written by the previous kernel (per-launch Q8_0 dequantisation): no weight loads before the dependency wait
    int multicast = 1;            // allow A-tile multicast over clusters of 4 CTAs along N (experimental, only with NSB_MC=1: measured slower)
    int a_fold = 0;               // 3xTF32 (fp32 operands on the tensor cores, launch_gemm_tc with OUT_F32 inputs): K = 3 a_fold, W = [hi | lo | hi], A = [hi | lo] (lda >= 2 a_fold)
    int rotate = 1;               // CTA n starts its k loop at k-block (n mod nk): de-synchronises the A-tile reads of the grid
};
void launch_gemm_simt(const GemmArgs& a, cudaStream_t st);
// Q8_0 x Q8_0 with the reference's arithmetic (gemm_q8_strict.cu): quantises the f32 rows of A into `scratch`, then integer block dots
void launch_gemm_q8_strict(const GemmArgs& a, void* scratch, size_t scratch_bytes, cudaStream_t st);
size_t q8_strict_scratch_bytes(int rows, int K);

// ---------------------------------------------------------------- layer kernels (kernels_layer.cu)
// Pending split-K reduction folded into a LayerNorm kernel: x += alpha * sum_s part[s] (fixed order => deterministic)
struct PartialSum { const float* part = nullptr; int n = 0; float alpha = 0.f; };
void launch_layernorm(float* x, int rows, const float* g, const float* b, void* y, int out_type, const PartialSum& ps, cudaStream_t st);
// y1 = LN(x; g1,b1) written back to x (f32) AND y2 = LN(y1; g2,b2) written as out_type  (norm_out fused with next norm_ff1)
void launch_layernorm2(float* x, int rows, const float* g1, const float* b1, const float* g2, const float* b2, void* y2,
                       int out_type, const PartialSum& ps, cudaStream_t st);

struct AttnArgs {
    const float* qkv;             // [planes][M][3072] f32 (q | k | v); planes > 1 = split-K partials of the QKV GEMM, summed on load
    int planes = 1; long long plane_stride = 0;   // elements between planes
    void* k_ring; void* v_ring;   // layer base; element (slot, r, c) at slot*slot_stride + r*1024 + c
    long long slot_stride;        // elements
    int kv_dtype;                 // 0 f32, 1 f16, 2 bf16
    const void* pos_proj;         // [L + 2T - 1][1024] in the K/V ring dtype, row = rel + (T-1)
    const float* bias_u; const float* bias_v;   // [1024]
    void* ctx; int out_type;      // [M][1024]
    const int* slot_of_b; const int* ring_pos; const int* valid_len;
    int B, T;
};
void launch_attention(const AttnArgs& a, cudaStream_t st);
// Full-context rel-pos attention of the non-streaming batch path (build_rel_pos_mha, nemo-ggml.cpp:591-680): one utterance,
// T frames, every query sees every key, no cache. qkv [T][3072] f32 (q | k | v); pos_proj rows in the K/V dtype with row
// (rel + pos_center) <-> relative position rel = query - key in [-(T-1), T-1]; ctx [T][1024] in out_type.
struct AttnFullArgs {
    const float* qkv; const void* pos_proj; int pos_center; int kv_dtype;
    const float* bias_u; const float* bias_v; void* ctx; int out_type; int T;
};
void launch_attention_full(const AttnFullArgs& a, cudaStream_t st);
void launch_dequant_q8(const void* q, const void* scales, void* out_f16, int N, int K, cudaStream_t st, int q4 = 0);   // gemm_tc.cu (q4: Q4_0 nibble plane)
bool pair_gemm_enabled();         // gemm_tc.cu: CTA-pair tiles on (default) / off (NSB_PAIR_GEMM=0)
bool q8_pair256_enabled();        // gemm_tc.cu: Q8_0 / Q4_0 dequantisation fused into the 256-row CTA-pair tiles at large batches: NSB_Q8_PAIR=1 (default off: the layer-ahead fp16 shadows are faster)

struct ConvModArgs {
    const float* pw1;             // [planes][M][2048] f32  (a | gate); planes > 1 = split-K partials of the pointwise GEMM, summed on load
    int planes = 1; long long plane_stride = 0;
    float* conv_cache;            // layer base; (slot, parity, r, c) at slot*slot_stride + parity*par_stride + r*1024 + c, r in 0..7
    long long slot_stride;
    // the state is double-buffered per slot: a step reads parity cc_par[slot] and writes the other one (every frame of the chunk is its
    // own CTA: the writer must not overwrite what CTAs of earlier frames still read); launch_advance_streams flips the parity
    const int* cc_par; long long par_stride;
    const float* dw_w;            // [9][1024] tap-major (GGUF layout)
    const float* ln_g; const float* ln_b;
    void* out; int out_type;      // [M][1024]
    const int* slot_of_b; int B, T;
};
void launch_conv_module(const ConvModArgs& a, cudaStream_t st);

void launch_advance_streams(const int* slot_of_b, int B, int T, int* ring_pos, int* valid_len, int* cc_par, cudaStream_t st);

// ---------------------------------------------------------------- RNN-T decode (kernels_decode.cu)
struct DecodeWeights {
    const float* embed;                       // [1025][640]
    const float* w_ih[2]; const float* w_hh[2]; const float* b_ih[2]; const float* b_hh[2];   // [2560][640], [2560]
    const float* pred_w; const float* pred_b; // [640][640], [640]
    const float* out_w; const float* out_b;   // [1025][640], [1025]
};
struct DecodeState {                          // slot-indexed, device
    float* hbuf; float* cbuf;                 // [S][2 parities][2 layers * 640]: committed state at parity par[slot], candidate at the other
    int* par;                                 // [S]
    float* dec_proj;                          // [S][640] joint.pred projection of the candidate
    int* prev_token; int* cand_valid;         // [S]
};
struct DecodeArgs {
    DecodeWeights w; DecodeState s;
    const float* enc_proj;                    // [B*T][640] (joint.enc applied, bias included)
    const int* slot_of_b; int B, T;
    int* out_tokens; int* out_count;          // [B][MAX_SYMBOLS*T], [B]
    int* out_frames;                          // optional [B][MAX_SYMBOLS*T]: encoder frame (within this call's T) each token was emitted at (timed_token::frame_idx)
    unsigned* barrier; unsigned long long* best;   // filled by launch_decode from its sync buffer
    int pipe_min_n;                           // filled by launch_decode: streams per phase from which the full-width grid uses the pipelined tiles
    float* logits_tap; int logits_tap_cap; int* logits_tap_n;   // optional: logits of batch row 0 per evaluation
};
// persistent kernel; sync_buf holds decode_sync_bytes(B) bytes. narrow_ctas = 0: one CTA per SM (cooperative launch); > 0: that many CTAs
// as CTA pairs, sharing the GPU with other kernels (decode overlap). pipe_min_n > 0 replaces the default streams-per-phase threshold of
// the pipelined tiles on a wide grid (operator tests). Returns the grid size used
int launch_decode(const DecodeArgs& a, void* sync_buf, cudaStream_t st, int narrow_ctas = 0, int pipe_min_n = 0);
int decode_narrow_ctas();          // NSB_DECODE_CTAS, default 20 (148 SMs - the 128 CTAs of the widest small-batch encoder kernel)
size_t decode_sync_bytes(int B);

}  // namespace nsb
