// engine.h -- per-GPU streaming engine (internal). Public face: include/nsb200.h
#pragma once
#include <deque>
#include <map>
#include <memory>
#include <string>
#include <tuple>
#include <vector>

#include "../../include/nsb200.h"
#include "gguf_loader.h"
#include "host_stream.h"
#include "kernels.cuh"

namespace nsb {

struct DevBuf {
    void* p = nullptr; size_t bytes = 0;
    DevBuf() = default;
    DevBuf(const DevBuf&) = delete; DevBuf& operator=(const DevBuf&) = delete;
    DevBuf(DevBuf&& o) noexcept : p(o.p), bytes(o.bytes) { o.p = nullptr; o.bytes = 0; }
    DevBuf& operator=(DevBuf&& o) noexcept { if (this != &o) { if (p) cudaFree(p); p = o.p; bytes = o.bytes; o.p = nullptr; o.bytes = 0; } return *this; }
    ~DevBuf() { if (p) cudaFree(p); }
    void alloc(size_t n, bool zero = true) {
        if (p) { cudaFree(p); p = nullptr; }
        bytes = n; if (!n) return;
        NSB_CUDA(cudaMalloc(&p, n));
        if (zero) { NSB_CUDA(cudaMemset(p, 0, n)); NSB_CUDA(cudaDeviceSynchronize()); }   // legacy-stream memset must not race the engine stream
    }
    template <class T> T* as() const { return (T*)p; }
};

constexpr int SNAP_BULK = 6;   // bulk device sections of a stream snapshot (stream_state.cu)

// a buffer that is not a valid stream snapshot (nsb_stream_import: NSB_ERR_FORMAT)
struct FormatError : std::runtime_error { using std::runtime_error::runtime_error; };

struct HostPinned {
    void* p = nullptr; size_t bytes = 0;
    ~HostPinned() { if (p) cudaFreeHost(p); }
    void alloc(size_t n) { if (p) { cudaFreeHost(p); p = nullptr; } bytes = n; if (n) NSB_CUDA(cudaMallocHost(&p, n)); }
    template <class T> T* as() const { return (T*)p; }
};

// one GEMM weight in the engine's compute arithmetic
struct Weight {
    std::string name; int n_out = 0, n_in = 0;
    int q4 = 0;             // Q8_0 mode, Q4_0 file: `data` is the nibble plane [n_out][n_in / 2] (fused-dequant GEMM variant)
    int shadow_slot = -1;   // Q8_0 mode: which of the layer's 8 matrices this is (offset into the fp16 shadow of the layer, see Engine::shadow_)
    bool f32 = false;       // kept in F32 by every GGUF (stem 1x1 convs and projection, joint.enc): Engine::gemm_f32w
    DevBuf data;            // f32 / f16 / bf16 [n_out][n_in]; Q8_0 mode: int8 quants [n_out][n_in]
    DevBuf scales;          // Q8_0 mode only: fp16 block scales [n_out][n_in / 32]
};

struct LayerW {
    DevBuf ln[10];          // ff1 g,b | attn g,b | conv g,b | ff2 g,b | out g,b
    Weight ff1a, ff1b, qkv, out, pw1, pw2, ff2a, ff2b;
    DevBuf bias_u, bias_v, dw_w, cln_g, cln_b;
    DevBuf pos_proj;        // [L+2T-1][1024] in the K/V ring dtype
};

class Engine {
public:
    Engine(const std::string& gguf_path, const nsb_engine_config& cfg);
    ~Engine();

    int open_stream(); void close_stream(int s); void reset_stream(int s);
    void push_pcm(int s, const int16_t* pcm, int n);
    bool ready(int s) const;
    int step();                       // returns #streams advanced
    // split form of step(): begin stages the ready streams' PCM, enqueues H2D + the step graph + D2H and returns at once
    // (the host can push the next chunk meanwhile); end waits for the OLDEST step in flight and hands its tokens to the
    // per-stream queues. Up to two steps may be in flight (begin, begin, end, begin, end, ...): the device then goes from one
    // step straight into the next.
    int step_begin();                 // returns #streams in the launched step (0 = nothing ready); throws with two steps in flight
    int step_end();                   // returns #streams advanced (0 = no step in flight)
    int pop_tokens(int s, int32_t* out, int cap);
    int chunks(int s) const;
    // stream snapshots (stream_state.cu; format in DESIGN.md §11): export leaves the stream open and unchanged, returns the bytes
    // written (out == nullptr: the size only); import takes the lowest free slot and returns it
    long long export_stream(int s, void* out, size_t cap);
    int import_stream(const void* blob, size_t bytes);
    std::string detok(const int32_t* t, int n) const;

    void bench_prepare(int n_streams, const int16_t* pcm, int samples_per_stream, int warm_chunks);
    float bench_step();
    // n steps enqueued back to back (no host synchronisation in between: the launch of step i+1 overlaps step i), one event
    // between consecutive steps; ms_each[i] = device time of step i, returns the total (first event -> last event)
    float bench_steps(int n, float* ms_each);
    // one bench step with every launch bracketed by CUDA events; per-class device ms and launch counts
    enum { PC_MEL = 0, PC_SUBSAMPLE, PC_LAYERNORM, PC_GEMM, PC_ATTENTION, PC_CONVMOD, PC_DECODE, PC_MISC, PC_COUNT };
    float bench_profile(float* ms_per_class, int* launches_per_class);
    // tuning: `iters` passes over all layers of one weight kind (0 ff1a,1 ff1b,2 qkv,3 out,4 pw1,5 pw2) with a forced tile config;
    // returns mean device us per GEMM
    float bench_gemm(int kind, int rows, int bn, int stages, int splits, int rotate, int iters);

    // device tracing (common.cuh): cap records; fetch copies the records written so far (launch order) and resets the counter
    void trace_enable(int cap);
    int trace_fetch(TraceRec* out, int cap);

    void set_cuda_graph(bool on) { collect_all(); cfg_.use_cuda_graph = on ? 1 : 0; }
    void debug_enable(bool on);
    long long debug_get(const std::string& name, float* out, size_t cap);
    long long debug_get_cache(int stream, int which, int layer, float* out, size_t cap);
    long long op_logmel(const int16_t* pcm, int n_streams, int n_samples, float* out, size_t cap);
    long long op_gemm(const std::string& name, const float* x, int rows, float* y, size_t cap);
    long long op_gemm_ex(const nsb_gemm_op& op, const float* x, void* y, size_t y_bytes, long long* guard_bad);
    void op_decode(nsb_decode_op& op);
    void op_layernorm(const float* x, int rows, const float* planes, int n_planes, float alpha, const float* g1, const float* b1,
                      const float* g2, const float* b2, bool fused, int out_type, float* x_out, void* y);
    // Non-streaming batch path (nemo_encode, reference src/nemo-ggml.cpp:1467-1535) for one utterance: whole-utterance log-mel ->
    // un-chunked subsampling -> non-cached layers with full-context rel-pos attention -> greedy decode from a fresh decoder state.
    // Borrows one free stream slot (decoder / conv state); the activations live in a workspace of their own, grown to the longest
    // utterance seen (any engine, whatever max_streams, takes up to 2048 encoder frames).
    // Returns the number of tokens (copies min(n, cap)); *n_frames = encoder frames; enc_out (optional) [frames][1024].
    long long transcribe_full(const int16_t* pcm, int n_samples, int32_t* tokens, int32_t* token_frames, int cap, int* n_frames, float* enc_out, size_t enc_cap);

    // facts
    int n_layers = 0, T = 1, R = 0, compute = NSB_COMPUTE_F32, kv_dtype = NSB_KV_F32, max_streams = 0;
    uint64_t fingerprint = 0;         // model identity a snapshot carries (GgufFile::fingerprint)
    std::vector<char> vocab;
    nsb_stats stats{};
    int chunk_samples() const { return (PRE_CACHE + 8 * T) * HOP; }
    int shift_samples() const { return 8 * T * HOP; }

private:
    void load_weights(const GgufFile& g);
    void upload_weight(Weight& w, const std::string& name, const std::vector<float>& host, int n_out, int n_in);
    // per-layer matrix straight from the file: Q8_0 tensors keep their quants in Q8_0 compute mode (fused-dequant GEMM)
    void load_layer_matrix(Weight& w, const GgufFile& g, const std::string& out_name, const std::vector<std::string>& parts, int n_out, int n_in);
    void alloc_state();
    void stream_upload(void* dst, const uint8_t* src, size_t bytes);   // mmap -> pinned chunks -> async H2D on st_
    HostPinned up_[2]; cudaEvent_t up_ev_[2] = {nullptr, nullptr}; int up_k_ = 0; DevBuf d_raw_;   // load-time staging
    void release_handles();            // graphs, events, stream (destructor and failed constructor)
    void zero_slot(int slot);
    void build_pos_tables(const GgufFile& g);
    void ensure_full_pos(int frames);  // positional projections for relative positions -(cap-1) .. cap-1 of the batch path, built on first use
    std::string gguf_path_;
    std::vector<DevBuf> full_pos_; int full_pos_cap_ = 0;
    void gemm(const void* A, long long lda, const Weight& W, int M, const float* bias, void* C, long long ldc, int epi, float alpha,
              int out_type);
    void gemm(GemmArgs& a, const Weight& W);   // the launch behind gemm() for explicit GemmArgs (A, M, C, epilogue set by the caller)
    // x += alpha * A W^T. Small batches: split-K into the workspace, reduction folded into the next LayerNorm (pending_).
    void gemm_residual(const void* A, long long lda, const Weight& W, int M, float* x, float alpha);
    bool split_consumers(int rows) const;
    // operator entry points (op_gemm, op_gemm_ex): weight by name, A operand as the step's producers leave it, split scratch of F32 matrices
    const Weight& op_weight(const std::string& name) const;
    const void* op_operand(const Weight& W, const float* xh, int rows, DevBuf& dx, DevBuf& da);
    struct SplitScratch;
    void q8_predequant(const Weight& W, int M, GemmArgs& a);
    void gemm_f32w(GemmArgs& g, const Weight& W, bool a_presplit);   // matrices kept in F32 by every GGUF: SIMT fp32 / 3xTF32
    void gemm_planes(const void* A, long long lda, const Weight& W, int M, void* C, int planes);
    PartialSum pending_{};
    // Everything between PCM-in-HBM and tokens-in-HBM, in two halves: the encoder (log-mel ... joint.enc projections) and the RNN-T
    // decode kernel. `side` selects one of two sets of hand-over buffers (stream slots of the batch, joint.enc projections, token ids).
    void run_encoder_kernels(int B, const int16_t* d_pcm, int side);
    void run_decode_kernels(int B, int side, cudaStream_t s, bool narrow);
    // Each half through a CUDA graph captured once per (batch size, PCM buffer, side): the ~350 launches of a step become two
    // cudaGraphLaunch calls (cfg.use_cuda_graph; bypassed while debug taps or per-launch profiling are on).
    // Decode overlap (small batches): the decode of step i runs on its own stream, on a handful of SMs, UNDER the encoder of step
    // i + 1 -- its per-symbol rounds are latency-bound and need no more, while the encoder's kernels at <= 128 token rows launch
    // <= 128 CTAs and leave those SMs idle anyway. Same kernel, same arithmetic, same tokens; the sides are what makes it safe.
    void join_decode_stream();                               // st_ waits for whatever the decode stream still runs
    int side_acquire();                                      // next side; orders st_ behind the decode that last read its buffers
    // pipelined = another step is (or is about to be) in flight behind this one: only then does the overlap buy anything -- a step
    // run on its own gets the full-width decode, which is the faster of the two in isolation. Returns the stream the step's tokens
    // become available on.
    cudaStream_t run_step(int B, const int16_t* d_pcm, int side, bool pipelined);
    bool overlap_decode(int rows, bool pipelined) const;
    struct StepGraph { cudaGraphExec_t exec = nullptr; long long launches = 0; };
    std::map<std::tuple<int, const void*, int>, StepGraph> graphs_;      // encoder halves
    std::map<std::tuple<int, int, int>, StepGraph> dec_graphs_;           // decode halves: (batch, side, narrow)
    template <class Key, class Fn> void run_graphed(std::map<Key, StepGraph>& cache, const Key& key, cudaStream_t s, Fn&& body);
    struct Side { DevBuf slot, encp, out_tok, out_cnt, sync; cudaEvent_t enc_done = nullptr, dec_done = nullptr; bool dec_pending = false; };
    static constexpr int MAX_INFLIGHT = 3;   // steps between step_begin and step_end: host-side step state and the device-side hand-over buffers are rings of this depth
    Side side_[MAX_INFLIGHT]; int side_next_ = 0;
    cudaStream_t st_dec_ = nullptr;
    cudaStream_t st_copy_ = nullptr;   // host -> device upload of a step's PCM rows: not on the engine stream, where it would sit between two steps' kernels
    struct StepIO {                   // host side of one step in flight
        HostPinned h_pcm, h_slot, h_tok, h_cnt;
        DevBuf d_pcm;                 // this step's PCM rows in HBM (uploaded on the copy stream while earlier steps compute)
        cudaEvent_t ev0 = nullptr, ev1 = nullptr, done = nullptr, h2d = nullptr;
        std::vector<int> batch;       // batch row -> stream slot
    };
    StepIO io_[MAX_INFLIGHT]; int io_next_ = 0, n_inflight_ = 0;
    void collect_tokens(StepIO& io);
    void collect_all();               // step_end() until nothing is in flight
    // strict modes keep every activation in f32 and run no tcgen05 kernel: NSB_COMPUTE_F32 (f32 weights, SIMT) and
    // NSB_COMPUTE_Q8_0_STRICT (the reference's Q8_0 x Q8_0 block arithmetic for the per-layer matrices, SIMT f32 for the rest)
    bool strict() const { return compute == NSB_COMPUTE_F32 || compute == NSB_COMPUTE_Q8_0_STRICT; }
    bool q8_planes_mode() const { return compute == NSB_COMPUTE_Q8_0 || compute == NSB_COMPUTE_Q8_0_STRICT; }
    int act_type() const { return strict() ? OUT_F32 : (compute == NSB_COMPUTE_BF16 ? OUT_BF16 : OUT_F16); }
    size_t act_size() const { return strict() ? 4 : 2; }
    void ensure_q8s_scratch(int rows);       // activation-quantiser scratch of the strict Q8_0 GEMM (never called inside a graph capture)
    void count_launch(int n = 1) { stats.kernel_launches += n; }

    nsb_engine_config cfg_{};
    int device_ = 0;
    cudaStream_t st_ = nullptr;
    cudaEvent_t ev0_ = nullptr, ev1_ = nullptr;

    // ---- weights ----
    std::vector<LayerW> layers_;
    std::map<std::string, Weight*> named_;   // for op_gemm
    DevBuf window_, cos_t_, sin_t_, fb_t_;
    DevBuf c0_w_, c0_b_, c2_w_, c2_b_, c3_b_, c5_w_, c5_b_, c6_b_, out_b_;
    Weight c3_w_, c6_w_, sub_out_w_;         // always f32: .data plain (SIMT strict mode), .scales = 3xTF32 split copy [hi | lo | hi] (tensor-core modes)
    Weight joint_enc_w_; DevBuf joint_enc_b_;
    DevBuf embed_, lstm_w_[4], lstm_b_[4], pred_w_, pred_b_, jout_w_, jout_b_;

    // ---- per-slot state ----
    DevBuf kv_;                    // [S][layers][2][L+T][1024] kv dtype
    DevBuf conv_cache_, cc_par_;   // conv state [S + 1][2 parities][layers][8][1024] f32, current parity [S + 1] (kernels.cuh: ConvModArgs)
    DevBuf mel_hist_;              // [S][9][128]
    DevBuf ring_pos_, valid_len_;  // [S] int
    DevBuf dec_h_, dec_c_, dec_par_, dec_proj_, prev_token_, cand_valid_;
    std::vector<HostStream> hs_;
    // snapshots: the slot's bulk arrays as (device pointer, bytes) in snapshot order; returns their total
    size_t snapshot_sections(int s, void** ptr, size_t* bytes) const;
    uint64_t device_checksum(void* const* ptr, const size_t* bytes, size_t first_word);   // syncs st_
    DevBuf snap_sum_;

    // ---- step workspace (batch-compact) ----
    int rl_ = 0;                   // PCM row length per stream-step
    DevBuf d_slot_, mel_new_, dw_, pw_, a3_, x_, a_, big_, qkv_, pw1_, encp_, part_;
    DevBuf out_tok_, out_cnt_, dec_sync_;
    // workspace of the non-streaming batch path (swapped in for the duration of transcribe_full)
    struct BatchWork { DevBuf dw, pw, a3, x, a, big, qkv, pw1, encp, part, out_tok, out_frm; int rows = 0; } bw_;
    void ensure_batch_work(int rows, int t2);
    void swap_batch_work();
    int consumer_planes_ = 1;         // planes the qkv_ / pw1_ buffers were sized for (split-K partials summed by the consumer kernels)

    // ---- bench ----
    DevBuf q8s_scratch_;              // strict Q8_0: int8 rows + block scales of the A operand of one GEMM
    // Q8_0 mode, large batches (>= 512 token rows: tensor-bound, every m-tile CTA of the fused kernel would repeat the dequantisation of
    // the same weight tile): the layer's 8 matrices are dequantised ONE LAYER AHEAD on a side stream into one of two fp16 shadows
    // (46 MB each), under the previous layer's kernels; HBM keeps holding (and streaming) the Q8_0 planes only.
    DevBuf shadow_[2]; size_t shadow_off_[8] = {}; size_t shadow_bytes_ = 0;
    cudaStream_t st_deq_ = nullptr; std::vector<cudaEvent_t> ev_deq_, ev_lstart_;
    const char* cur_shadow_ = nullptr;                       // shadow of the layer whose GEMMs are being launched (nullptr: not in shadow mode)
    bool shadow_mode(int rows) const;
    void dequant_layer_async(int l, cudaStream_t s);
    DevBuf wscratch_;                 // fp16 copy of ONE Q8_0 matrix (large batches), rewritten before every GEMM that uses it
    DevBuf bench_pcm_; int bench_B_ = 0, bench_n_ = 1; long long bench_i_ = 0;   // [bench_n_][bench_B_][rl_] staged chunks, cycled
    const int16_t* bench_next_pcm();
    // ---- per-launch profiling (bench_profile only) ----
    struct ProfRec { int cls; cudaEvent_t a, b; };
    bool profiling_ = false; std::vector<ProfRec> prof_; std::vector<cudaEvent_t> ev_pool_; size_t ev_used_ = 0;
    cudaEvent_t prof_event();
    struct ProfScope {
        Engine* e; cudaEvent_t b = nullptr;
        ProfScope(Engine* e_, int cls) : e(e_) {
            if (!e->profiling_) return;
            cudaEvent_t a = e->prof_event(); b = e->prof_event();
            cudaEventRecord(a, e->st_); e->prof_.push_back({cls, a, b});
        }
        ~ProfScope() { if (b) cudaEventRecord(b, e->st_); }
    };

    // ---- debug taps ----
    bool debug_ = false; int dbg_B_ = 0, last_B_ = 0;
    DevBuf dbg_mel_, dbg_sub_, dbg_layers_, dbg_logits_, dbg_logits_n_;
    DevBuf trace_; int trace_cap_ = 0;
};

}  // namespace nsb
