// c_api.cu -- extern "C" face of the engine (include/nsb200.h). Exceptions never cross the boundary.
#include <algorithm>
#include <cstring>
#include <string>

#include <cuda_profiler_api.h>

#include "engine.h"

using nsb::Engine;

struct nsb_engine { Engine* impl; };

static thread_local std::string g_err;
static int fail(int code, const std::string& msg) { g_err = msg; return code; }

#define NSB_TRY try {
#define NSB_CATCH                                                                         \
    } catch (const nsb::CudaError& e) { return fail(NSB_ERR_CUDA, e.what());              \
    } catch (const std::invalid_argument& e) { return fail(NSB_ERR_ARG, e.what());        \
    } catch (const nsb::FormatError& e) { return fail(NSB_ERR_FORMAT, e.what());          \
    } catch (const std::bad_alloc&) { return fail(NSB_ERR_NOMEM, "out of host memory");   \
    } catch (const std::exception& e) { return fail(NSB_ERR_STATE, e.what()); }

extern "C" {

const char* nsb_last_error(void) { return g_err.c_str(); }

int nsb_gguf_probe(const char* path, nsb_model_info* info) {
    if (!path || !info) return fail(NSB_ERR_ARG, "null argument");
    try {
        nsb::GgufFile g; g.open(path);
        memset(info, 0, sizeof(*info));
        auto u = [&](const char* k, int def) { auto it = g.u32.find(k); return it == g.u32.end() ? def : (int)it->second; };
        info->n_mels = u("nemo.n_mels", 128); info->d_model = u("nemo.d_model", 1024); info->n_heads = u("nemo.n_heads", 8);
        info->d_head = u("nemo.d_head", 128); info->d_ff = u("nemo.d_ff", 4096); info->n_layers = u("nemo.n_layers", 24);
        info->kernel_size = u("nemo.kernel_size", 31); info->vocab_size = u("nemo.vocab_size", 1025);
        info->decoder_dim = u("nemo.decoder_dim", 320); info->joint_dim = u("nemo.joint_dim", 640);
        info->n_tensors = (int)g.tensors.size();
        auto it = g.tensors.find("encoder.layers.0.feed_forward1.linear1.weight");
        info->weight_type = it == g.tensors.end() ? 0 : it->second.type;
        memcpy(info->vocab, g.vocab_raw.data(), std::min(g.vocab_raw.size(), sizeof(info->vocab)));
        for (const char* need : {"encoder.pre_encode.conv.0.weight", "encoder.pre_encode.out.weight", "decoder.prediction.embed.weight",
                                 "joint.enc.weight", "joint.joint_net.2.weight", "preprocessor.featurizer.fb", "preprocessor.featurizer.window"})
            g.require(need);                                    // the reference's "missing tensor" check (nemo-ggml.cpp:362-384)
        return NSB_OK;
    } catch (const std::exception& e) {
        const std::string m = e.what();
        return fail(m.find("cannot open") != std::string::npos ? NSB_ERR_IO : NSB_ERR_FORMAT, m);
    }
}

long long nsb_gguf_read_tensor(const char* path, const char* name, float* out, size_t cap, int* type) {
    if (!path || !name) return fail(NSB_ERR_ARG, "null argument");
    try {
        nsb::GgufFile g; g.open(path);
        const nsb::GgufTensor& t = g.require(name);
        if (type) *type = t.type;
        const long long n = (long long)t.n_elements();
        if (!out) return n;                                   // query: element count only
        if ((size_t)n > cap) return fail(NSB_ERR_ARG, "nsb_gguf_read_tensor: buffer too small for " + std::to_string(n) + " elements");
        const std::vector<float> v = g.read_dequant(name);
        memcpy(out, v.data(), v.size() * sizeof(float));
        return n;
    } catch (const std::exception& e) {
        const std::string m = e.what();
        return fail(m.find("cannot open") != std::string::npos ? NSB_ERR_IO : NSB_ERR_FORMAT, m);
    }
}

void nsb_default_config(nsb_engine_config* c) {
    if (!c) return;
    memset(c, 0, sizeof(*c));
    c->device = 0; c->compute = NSB_COMPUTE_AUTO; c->kv_dtype = NSB_KV_F32; c->att_right_context = 0;   // default_config(): pure causal (nemo-stream.h:103-105)
    c->max_streams = 1; c->use_cuda_graph = 1;
}

int nsb_engine_create(const char* path, const nsb_engine_config* cfg, nsb_engine** out) {
    if (!path || !out) return fail(NSB_ERR_ARG, "null argument");
    *out = nullptr;
    nsb_engine_config c; if (cfg) c = *cfg; else nsb_default_config(&c);
    try {
        Engine* e = new Engine(path, c);
        *out = new nsb_engine{e};
        return NSB_OK;
    } catch (const nsb::CudaError& e) { return fail(NSB_ERR_CUDA, e.what());
    } catch (const std::invalid_argument& e) { return fail(NSB_ERR_ARG, e.what());
    } catch (const std::exception& e) {
        const std::string m = e.what();
        return fail(m.find("cannot open") != std::string::npos ? NSB_ERR_IO : NSB_ERR_FORMAT, m);
    }
}
void nsb_engine_destroy(nsb_engine* e) { if (e) { delete e->impl; delete e; } }

int nsb_engine_n_layers(const nsb_engine* e) { return e ? e->impl->n_layers : NSB_ERR_ARG; }
int nsb_engine_vocab_size(const nsb_engine* e) { return e ? nsb::VOCAB : NSB_ERR_ARG; }
const char* nsb_engine_vocab(const nsb_engine* e) { return e ? e->impl->vocab.data() : nullptr; }
int nsb_engine_chunk_samples(const nsb_engine* e) { return e ? e->impl->chunk_samples() : NSB_ERR_ARG; }
int nsb_engine_shift_samples(const nsb_engine* e) { return e ? e->impl->shift_samples() : NSB_ERR_ARG; }
int nsb_engine_compute(const nsb_engine* e) { return e ? e->impl->compute : NSB_ERR_ARG; }

int nsb_engine_set_cuda_graph(nsb_engine* e, int on) { if (!e) return fail(NSB_ERR_ARG, "null engine"); NSB_TRY e->impl->set_cuda_graph(on != 0); return NSB_OK; NSB_CATCH }

int nsb_stream_open(nsb_engine* e) { if (!e) return fail(NSB_ERR_ARG, "null engine"); NSB_TRY return e->impl->open_stream(); NSB_CATCH }
int nsb_stream_close(nsb_engine* e, int s) { if (!e) return fail(NSB_ERR_ARG, "null engine"); NSB_TRY e->impl->close_stream(s); return NSB_OK; NSB_CATCH }
int nsb_stream_reset(nsb_engine* e, int s) { if (!e) return fail(NSB_ERR_ARG, "null engine"); NSB_TRY e->impl->reset_stream(s); return NSB_OK; NSB_CATCH }
long long nsb_stream_export(nsb_engine* e, int s, void* out, size_t cap) {
    if (!e) return fail(NSB_ERR_ARG, "null engine"); NSB_TRY return e->impl->export_stream(s, out, cap); NSB_CATCH }
int nsb_stream_import(nsb_engine* e, const void* snapshot, size_t bytes) {
    if (!e || !snapshot) return fail(NSB_ERR_ARG, "bad argument"); NSB_TRY return e->impl->import_stream(snapshot, bytes); NSB_CATCH }
int nsb_stream_push_pcm(nsb_engine* e, int s, const int16_t* pcm, int n) {
    if (!e) return fail(NSB_ERR_ARG, "null engine"); NSB_TRY e->impl->push_pcm(s, pcm, n); return NSB_OK; NSB_CATCH }
int nsb_push_pcm_batch(nsb_engine* e, int n_streams, const int32_t* streams, const int16_t* pcm, int row_stride, int n_samples) {
    if (!e || !streams || (!pcm && n_samples > 0) || n_streams < 0) return fail(NSB_ERR_ARG, "bad argument");
    NSB_TRY for (int i = 0; i < n_streams; ++i) e->impl->push_pcm(streams[i], pcm + (size_t)i * row_stride, n_samples); return NSB_OK; NSB_CATCH }
int nsb_pop_tokens_batch(nsb_engine* e, int n_streams, const int32_t* streams, int32_t* out, int cap_per_stream, int32_t* counts) {
    if (!e || !streams || !out || !counts || cap_per_stream < 0) return fail(NSB_ERR_ARG, "bad argument");
    NSB_TRY int total = 0;
    for (int i = 0; i < n_streams; ++i) { counts[i] = e->impl->pop_tokens(streams[i], out + (size_t)i * cap_per_stream, cap_per_stream); total += counts[i]; }
    return total; NSB_CATCH }
int nsb_stream_ready(const nsb_engine* e, int s) { if (!e || s < 0 || s >= e->impl->max_streams) return NSB_ERR_ARG; return e->impl->ready(s) ? 1 : 0; }
int nsb_engine_step(nsb_engine* e) { if (!e) return fail(NSB_ERR_ARG, "null engine"); NSB_TRY return e->impl->step(); NSB_CATCH }
int nsb_engine_step_begin(nsb_engine* e) { if (!e) return fail(NSB_ERR_ARG, "null engine"); NSB_TRY return e->impl->step_begin(); NSB_CATCH }
int nsb_engine_step_end(nsb_engine* e) { if (!e) return fail(NSB_ERR_ARG, "null engine"); NSB_TRY return e->impl->step_end(); NSB_CATCH }
int nsb_engine_drain(nsb_engine* e) {
    if (!e) return fail(NSB_ERR_ARG, "null engine");
    NSB_TRY int total = 0; for (;;) { int n = e->impl->step(); if (n <= 0) break; total += n; } return total; NSB_CATCH }
int nsb_stream_pop_tokens(nsb_engine* e, int s, int32_t* out, int cap) {
    if (!e || !out || cap < 0) return fail(NSB_ERR_ARG, "bad argument"); NSB_TRY return e->impl->pop_tokens(s, out, cap); NSB_CATCH }
int nsb_stream_chunks(const nsb_engine* e, int s) { if (!e) return NSB_ERR_ARG; NSB_TRY return e->impl->chunks(s); NSB_CATCH }

int nsb_detokenize(const nsb_engine* e, const int32_t* t, int n, char* out, int cap) {
    if (!e || (!t && n > 0) || !out) return fail(NSB_ERR_ARG, "bad argument");
    NSB_TRY const std::string r = e->impl->detok(t, n);
    if ((int)r.size() + 1 > cap) return -(int)r.size() - 1;
    memcpy(out, r.c_str(), r.size() + 1); return (int)r.size(); NSB_CATCH }

void nsb_engine_get_stats(const nsb_engine* e, nsb_stats* out) { if (e && out) *out = e->impl->stats; }

int nsb_bench_prepare(nsb_engine* e, int n, const int16_t* pcm, int sps, int warm) {
    if (!e || !pcm) return fail(NSB_ERR_ARG, "bad argument"); NSB_TRY e->impl->bench_prepare(n, pcm, sps, warm); return NSB_OK; NSB_CATCH }
int nsb_bench_step(nsb_engine* e, float* ms) {
    if (!e) return fail(NSB_ERR_ARG, "null engine"); NSB_TRY const float t = e->impl->bench_step(); if (ms) *ms = t; return NSB_OK; NSB_CATCH }

int nsb_bench_steps(nsb_engine* e, int n, float* ms_each, float* total_ms) {
    if (!e) return fail(NSB_ERR_ARG, "null engine"); NSB_TRY const float t = e->impl->bench_steps(n, ms_each); if (total_ms) *total_ms = t; return NSB_OK; NSB_CATCH }

int nsb_bench_profile(nsb_engine* e, float* ms_per_class, int* launches_per_class, float* total_ms) {
    if (!e || !ms_per_class || !launches_per_class) return fail(NSB_ERR_ARG, "bad argument");
    NSB_TRY const float t = e->impl->bench_profile(ms_per_class, launches_per_class); if (total_ms) *total_ms = t; return NSB_OK; NSB_CATCH }

int nsb_bench_gemm(nsb_engine* e, int kind, int rows, int bn, int stages, int splits, int rotate, int iters, float* us) {
    if (!e || !us) return fail(NSB_ERR_ARG, "bad argument"); NSB_TRY *us = e->impl->bench_gemm(kind, rows, bn, stages, splits, rotate, iters); return NSB_OK; NSB_CATCH }

int nsb_trace_enable(nsb_engine* e, int capacity) { if (!e) return fail(NSB_ERR_ARG, "null engine"); NSB_TRY e->impl->trace_enable(capacity); return NSB_OK; NSB_CATCH }
int nsb_trace_fetch(nsb_engine* e, nsb_trace_record* out, int cap) {
    if (!e || (!out && cap > 0)) return fail(NSB_ERR_ARG, "bad argument");
    static_assert(sizeof(nsb_trace_record) == sizeof(nsb::TraceRec), "trace record layout");
    NSB_TRY return e->impl->trace_fetch(reinterpret_cast<nsb::TraceRec*>(out), cap); NSB_CATCH }

int nsb_profiler_range(int on) { return (on ? cudaProfilerStart() : cudaProfilerStop()) == cudaSuccess ? NSB_OK : NSB_ERR_CUDA; }

int nsb_debug_enable(nsb_engine* e, int on) { if (!e) return fail(NSB_ERR_ARG, "null engine"); NSB_TRY e->impl->debug_enable(on != 0); return NSB_OK; NSB_CATCH }
int nsb_debug_get(nsb_engine* e, const char* name, float* out, size_t cap) {
    if (!e || !name || !out) return fail(NSB_ERR_ARG, "bad argument"); NSB_TRY return (int)e->impl->debug_get(name, out, cap); NSB_CATCH }
int nsb_debug_get_cache(nsb_engine* e, int s, int which, int layer, float* out, size_t cap) {
    if (!e || !out) return fail(NSB_ERR_ARG, "bad argument"); NSB_TRY return (int)e->impl->debug_get_cache(s, which, layer, out, cap); NSB_CATCH }

int nsb_op_logmel(nsb_engine* e, const int16_t* pcm, int ns, int n, float* out, size_t cap) {
    if (!e || !pcm || !out) return fail(NSB_ERR_ARG, "bad argument"); NSB_TRY return (int)e->impl->op_logmel(pcm, ns, n, out, cap); NSB_CATCH }
int nsb_op_gemm(nsb_engine* e, const char* name, const float* x, int rows, float* y, size_t cap) {
    if (!e || !name || !x || !y) return fail(NSB_ERR_ARG, "bad argument"); NSB_TRY return (int)e->impl->op_gemm(name, x, rows, y, cap); NSB_CATCH }

int nsb_op_gemm_ex(nsb_engine* e, const nsb_gemm_op* op, const float* x, void* y, size_t y_bytes, long long* guard_bad) {
    if (!e || !op || !op->weight || !x || !y) return fail(NSB_ERR_ARG, "bad argument");
    NSB_TRY return (int)e->impl->op_gemm_ex(*op, x, y, y_bytes, guard_bad); NSB_CATCH }
int nsb_op_decode(nsb_engine* e, nsb_decode_op* op) {
    if (!e || !op) return fail(NSB_ERR_ARG, "bad argument");
    NSB_TRY e->impl->op_decode(*op); return NSB_OK; NSB_CATCH }
int nsb_op_layernorm(nsb_engine* e, const float* x, int rows, const float* planes, int n_planes, float alpha, const float* g1, const float* b1,
                     const float* g2, const float* b2, int fused, int out_type, float* x_out, void* y) {
    if (!e || !x || !x_out || !y) return fail(NSB_ERR_ARG, "bad argument");
    NSB_TRY e->impl->op_layernorm(x, rows, planes, n_planes, alpha, g1, b1, g2, b2, fused != 0, out_type, x_out, y); return NSB_OK; NSB_CATCH }

int nsb_transcribe_full(nsb_engine* e, const int16_t* pcm, int n, int32_t* tokens, int32_t* token_frames, int cap, int* n_frames, float* enc_out, size_t enc_cap) {
    if (!e || !pcm) return fail(NSB_ERR_ARG, "bad argument"); NSB_TRY return (int)e->impl->transcribe_full(pcm, n, tokens, token_frames, cap, n_frames, enc_out, enc_cap); NSB_CATCH }

}  // extern "C"
