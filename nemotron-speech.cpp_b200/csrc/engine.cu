// engine.cu -- host orchestration of the B200 streaming engine: weight residency, per-stream state in HBM,
// PCM staging, the batched per-chunk launch sequence, token hand-back.
//
// Replaces (reference, relative to its repo root):
//   nemo_model_load / nemo_init_with_backend             src/nemo-ggml.cpp:83-433
//   nemo_stream_context::init / nemo_encoder_graph::init src/nemo-stream.cpp:36-79, :257-302
//   nemo_stream_process_incremental + process_mel_chunk_streaming   src/nemo-stream.cpp:961-1134
// with one difference in shape: the reference handles ONE stream per context; this engine advances every
// stream that has a full chunk buffered in ONE batched step (B streams x T frames = B*T token rows per GEMM).
#include "engine.h"

#include <algorithm>
#include <cmath>
#include <cstddef>
#include <cstdlib>
#include <cstring>
#include <limits>

namespace nsb {

// implemented in gemm_tc.cu (tcgen05 / TMEM / TMA)
void launch_gemm_tc(const GemmArgs& a, int in_type /*OUT_F16 | OUT_BF16*/, cudaStream_t st);

constexpr int MAX_SPLITS = 8;
constexpr size_t SPLIT_CONSUMER_MAX_ROWS = 256;   // up to this many token rows per step the QKV / pointwise-1 GEMMs are split-K as well

bool tf32x3_enabled() {
    static const bool on = [] { const char* e = getenv("NSB_STEM_TF32"); return !(e && e[0] == '1'); }();
    return on;
}
bool pdl_enabled() {
    static const bool on = [] { const char* e = getenv("NSB_NO_PDL"); return !(e && e[0] == '1'); }();
    return on;
}

namespace {

__global__ void convert_kernel(const float* __restrict__ in, void* __restrict__ out, size_t n, int out_type) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        store_out(out, i, in[i], out_type);
}
void convert_to(const float* d_in, void* d_out, size_t n, int out_type, cudaStream_t st) {
    if (!n) return;
    int blocks = (int)std::min<size_t>((n + 255) / 256, 148 * 8);
    convert_kernel<<<blocks, 256, 0, st>>>(d_in, d_out, n, out_type);
}

// ---- load-time unpacking of raw GGUF tensor bytes ON THE DEVICE (the host only moves bytes: mmap -> pinned chunk -> async H2D) ----
// out[i] += sum of n_planes split-K planes (fixed order): the reduction of a split-K GEMM that no LayerNorm follows (joint.enc)
__global__ void __launch_bounds__(256) add_planes_kernel(float* __restrict__ out, const float* __restrict__ part, int n_planes, size_t plane, size_t n4) {
    NSB_KERNEL_PROLOGUE(TR_OTHER)
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n4) {
        float4 v = reinterpret_cast<const float4*>(out)[i];
        for (int z = 0; z < n_planes; ++z) {
            const float4 t = __ldcg(reinterpret_cast<const float4*>(part + (size_t)z * plane) + i);
            v.x += t.x; v.y += t.y; v.z += t.z; v.w += t.w;
        }
        reinterpret_cast<float4*>(out)[i] = v;
    }
    NSB_KERNEL_EPILOGUE();
}
__global__ void cvt_f16_kernel(const __half* __restrict__ in, void* __restrict__ out, size_t n, int out_type) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        store_out(out, i, __half2float(in[i]), out_type);           // fp16 -> f32 exact, then one rounding (bf16) like the host path
}
// Q8_0 blocks (fp16 d + 32 x int8, 34 bytes, 2-byte aligned) -> int8 plane + fp16 scale plane; one thread per block
__global__ void unpack_q8_planes_kernel(const uint16_t* __restrict__ raw, int8_t* __restrict__ q, uint16_t* __restrict__ d, size_t nb) {
    for (size_t b = (size_t)blockIdx.x * blockDim.x + threadIdx.x; b < nb; b += (size_t)gridDim.x * blockDim.x) {
        const uint16_t* p = raw + b * 17;
        uint32_t w[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) w[i] = (uint32_t)p[1 + 2 * i] | ((uint32_t)p[2 + 2 * i] << 16);
        d[b] = p[0];
        uint4* dst = reinterpret_cast<uint4*>(q + b * 32);
        dst[0] = make_uint4(w[0], w[1], w[2], w[3]); dst[1] = make_uint4(w[4], w[5], w[6], w[7]);
    }
}
// Q4_0 blocks (fp16 d + 16 nibble bytes, 18 bytes) -> nibble plane (16 bytes per block, as stored) + fp16 scale plane; strict = 1: int8
// plane of q - 8 instead (32 bytes per block: the strict Q8_0 x Q8_0 GEMM takes any int8 weight quants)
__global__ void unpack_q4_planes_kernel(const uint16_t* __restrict__ raw, uint8_t* __restrict__ q, uint16_t* __restrict__ d, size_t nb, int strict) {
    for (size_t b = (size_t)blockIdx.x * blockDim.x + threadIdx.x; b < nb; b += (size_t)gridDim.x * blockDim.x) {
        const uint16_t* p = raw + b * 9;
        uint32_t w[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) w[i] = (uint32_t)p[1 + 2 * i] | ((uint32_t)p[2 + 2 * i] << 16);
        d[b] = p[0];
        if (!strict) { *reinterpret_cast<uint4*>(q + b * 16) = make_uint4(w[0], w[1], w[2], w[3]); continue; }
        int8_t v[32];
#pragma unroll
        for (int i = 0; i < 16; ++i) { const uint32_t by = (w[i >> 2] >> (8 * (i & 3))) & 0xFFu; v[i] = (int8_t)((int)(by & 0xF) - 8); v[16 + i] = (int8_t)((int)(by >> 4) - 8); }
        uint4* dst = reinterpret_cast<uint4*>(q + b * 32);
        dst[0] = *reinterpret_cast<uint4*>(&v[0]); dst[1] = *reinterpret_cast<uint4*>(&v[16]);
    }
}
// Q8_0 / Q4_0 blocks -> dense values d * q (exact in f32), rounded once to out_type: what ggml's dequantize_row_* returns
__global__ void dequant_blocks_kernel(const uint16_t* __restrict__ raw, void* __restrict__ out, size_t nb, int q4, int out_type) {
    for (size_t b = (size_t)blockIdx.x * blockDim.x + threadIdx.x; b < nb; b += (size_t)gridDim.x * blockDim.x) {
        const uint16_t* p = raw + b * (q4 ? 9 : 17);
        const float d = __half2float(__ushort_as_half(p[0]));
        if (q4) {                                                   // byte i: element i = low nibble, element i + 16 = high nibble, value d * (q - 8)
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const uint32_t v = p[1 + i];
                store_out(out, b * 32 + 2 * i, d * (float)((int)(v & 0xF) - 8), out_type);
                store_out(out, b * 32 + 2 * i + 1, d * (float)((int)((v >> 8) & 0xF) - 8), out_type);
                store_out(out, b * 32 + 16 + 2 * i, d * (float)((int)((v >> 4) & 0xF) - 8), out_type);
                store_out(out, b * 32 + 16 + 2 * i + 1, d * (float)((int)(v >> 12) - 8), out_type);
            }
        } else {
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                const uint32_t v = p[1 + i];
                store_out(out, b * 32 + 2 * i, d * (float)(int8_t)(v & 0xFF), out_type);
                store_out(out, b * 32 + 2 * i + 1, d * (float)(int8_t)(v >> 8), out_type);
            }
        }
    }
}
int grid_for(size_t n) { return (int)std::min<size_t>((n + 255) / 256, 148 * 8); }

// any per-layer matrix as floats (F32 / F16 as stored, Q8_0 / Q4_0 dequantised): gguf_loader.cpp, pure host code tested on CPU
std::vector<float> read_matrix_f32(const GgufFile& g, const std::string& name) { return g.read_dequant(name); }

// Host -> device copy that is COMPLETE on return. cudaMemcpy from pageable memory may return while the DMA from the
// staging buffer is still in flight, and the engine's kernels run on a non-blocking stream that is not ordered after
// the legacy stream -- so every load-time / operator upload goes through here.
void h2d_sync(void* dst, const void* src, size_t bytes) {
    NSB_CUDA(cudaMemcpy(dst, src, bytes, cudaMemcpyHostToDevice));
    NSB_CUDA(cudaDeviceSynchronize());
}
void upload(DevBuf& d, const std::vector<float>& h) {
    d.alloc(h.size() * sizeof(float), false);
    h2d_sync(d.p, h.data(), h.size() * sizeof(float));
}

// 3xTF32 weight layout (common.cuh: split_tf32): [n_out][hi (K) | lo (K) | hi (K)], rounding = cvt.rna.tf32 (nearest, ties away)
float host_to_tf32(float v) {
    uint32_t u; memcpy(&u, &v, 4);
    if ((u & 0x7f800000u) == 0x7f800000u) return v;                 // inf / nan
    u = (u + 0x1000u) & ~0x1fffu;
    float r; memcpy(&r, &u, 4); return r;
}
std::vector<float> tf32x3_weight(const std::vector<float>& w, int n_out, int n_in) {
    std::vector<float> o((size_t)n_out * 3 * n_in);
    for (int n = 0; n < n_out; ++n)
        for (int k = 0; k < n_in; ++k) {
            const float v = w[(size_t)n * n_in + k], hi = host_to_tf32(v), lo = host_to_tf32(v - hi);
            float* r = &o[(size_t)n * 3 * n_in];
            r[k] = hi; r[n_in + k] = lo; r[2 * n_in + k] = hi;
        }
    return o;
}

// positional table row for relative position p (src/nemo-ggml.cpp:17-32)
void pos_emb_row(int p_int, float* row) {
    const float p = (float)p_int;
    for (int i = 0; i < D_MODEL; i += 2) {
        const float div_term = std::exp(-(float)i * std::log(10000.0f) / (float)D_MODEL);
        row[i] = std::sin(p * div_term);
        row[i + 1] = std::cos(p * div_term);
    }
}
}  // namespace

// ------------------------------------------------------------------------------------------
Engine::Engine(const std::string& path, const nsb_engine_config& cfg) : cfg_(cfg), gguf_path_(path) {
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        throw CudaError("no CUDA device available (this engine has no CPU fallback)");
    device_ = cfg.device;
    NSB_CUDA(cudaSetDevice(device_));
    cudaDeviceProp prop{};
    NSB_CUDA(cudaGetDeviceProperties(&prop, device_));
    if (prop.major != 10) throw CudaError(std::string("device '") + prop.name + "' is not sm_100 (kernels are built for sm_100a only)");
    try {
    NSB_CUDA(cudaStreamCreateWithFlags(&st_, cudaStreamNonBlocking));
    NSB_CUDA(cudaStreamCreateWithFlags(&st_dec_, cudaStreamNonBlocking));
    NSB_CUDA(cudaStreamCreateWithFlags(&st_copy_, cudaStreamNonBlocking));
    for (Side& sd : side_) { NSB_CUDA(cudaEventCreateWithFlags(&sd.enc_done, cudaEventDisableTiming)); NSB_CUDA(cudaEventCreateWithFlags(&sd.dec_done, cudaEventDisableTiming)); }
    NSB_CUDA(cudaEventCreate(&ev0_));
    NSB_CUDA(cudaEventCreate(&ev1_));
    for (StepIO& io : io_) { NSB_CUDA(cudaEventCreate(&io.ev0)); NSB_CUDA(cudaEventCreate(&io.ev1)); NSB_CUDA(cudaEventCreateWithFlags(&io.done, cudaEventDisableTiming));
                            NSB_CUDA(cudaEventCreateWithFlags(&io.h2d, cudaEventDisableTiming)); }

    R = cfg.att_right_context;
    if (R < 0 || R > 64) throw std::invalid_argument("att_right_context out of range");
    T = 1 + R;
    max_streams = std::max(1, cfg.max_streams);
    kv_dtype = cfg.kv_dtype;
    if (kv_dtype < 0 || kv_dtype > 2) throw std::invalid_argument("kv_dtype");

    GgufFile g;
    g.open(path);
    n_layers = g.u32.count("nemo.n_layers") ? (int)g.u32["nemo.n_layers"] : 24;
    const int vs = g.u32.count("nemo.vocab_size") ? (int)g.u32["nemo.vocab_size"] : VOCAB;
    if (vs != VOCAB) throw std::runtime_error("unsupported vocab_size (expected 1025)");
    // vocab: bounded copy + zero fill (the reference memcpy's vocab_size*8 bytes unconditionally, nemo-ggml.cpp:137-146)
    vocab.assign((size_t)VOCAB * 8, 0);
    memcpy(vocab.data(), g.vocab_raw.data(), std::min(g.vocab_raw.size(), vocab.size()));

    compute = cfg.compute;
    if (compute == NSB_COMPUTE_AUTO) {
        const int t = g.require("encoder.layers.0.feed_forward1.linear1.weight").type;
        // Q8_0 and Q4_0 files stay quantised in HBM (fused-dequant GEMM; NSB_COMPUTE_F16 on such a file expands it to fp16 at load)
        compute = t == GGML_F32 ? NSB_COMPUTE_F32 : t == GGML_F16 ? NSB_COMPUTE_F16 : NSB_COMPUTE_Q8_0;
    }
    fingerprint = g.fingerprint();
    load_weights(g);
    alloc_state();
    build_pos_tables(g);
    NSB_CUDA(cudaStreamSynchronize(st_));
    NSB_CUDA(cudaGetLastError());
    d_raw_ = DevBuf();                                             // load-time staging: released
    for (int i = 0; i < 2; ++i) { up_[i].alloc(0); if (up_ev_[i]) { cudaEventDestroy(up_ev_[i]); up_ev_[i] = nullptr; } }
    } catch (...) { release_handles(); throw; }                    // a throwing constructor runs no destructor: free the stream and events here
}

void Engine::release_handles() {
    cudaSetDevice(device_);
    cudaDeviceSynchronize();
    for (auto& g : graphs_) if (g.second.exec) cudaGraphExecDestroy(g.second.exec);
    graphs_.clear();
    for (auto& g : dec_graphs_) if (g.second.exec) cudaGraphExecDestroy(g.second.exec);
    dec_graphs_.clear();
    for (Side& sd : side_) { if (sd.enc_done) { cudaEventDestroy(sd.enc_done); sd.enc_done = nullptr; } if (sd.dec_done) { cudaEventDestroy(sd.dec_done); sd.dec_done = nullptr; } }
    if (st_dec_) { cudaStreamDestroy(st_dec_); st_dec_ = nullptr; }
    if (st_copy_) { cudaStreamDestroy(st_copy_); st_copy_ = nullptr; }
    for (cudaEvent_t e : ev_deq_) cudaEventDestroy(e);
    for (cudaEvent_t e : ev_lstart_) cudaEventDestroy(e);
    ev_deq_.clear(); ev_lstart_.clear();
    if (st_deq_) { cudaStreamDestroy(st_deq_); st_deq_ = nullptr; }
    for (cudaEvent_t e : ev_pool_) cudaEventDestroy(e);
    ev_pool_.clear();
    if (ev0_) { cudaEventDestroy(ev0_); ev0_ = nullptr; }
    if (ev1_) { cudaEventDestroy(ev1_); ev1_ = nullptr; }
    for (StepIO& io : io_) {
        if (io.ev0) { cudaEventDestroy(io.ev0); io.ev0 = nullptr; }
        if (io.ev1) { cudaEventDestroy(io.ev1); io.ev1 = nullptr; }
        if (io.done) { cudaEventDestroy(io.done); io.done = nullptr; }
        if (io.h2d) { cudaEventDestroy(io.h2d); io.h2d = nullptr; }
    }
    for (int i = 0; i < 2; ++i) if (up_ev_[i]) { cudaEventDestroy(up_ev_[i]); up_ev_[i] = nullptr; }
    if (st_) { cudaStreamDestroy(st_); st_ = nullptr; }
}

Engine::~Engine() { release_handles(); }

void Engine::upload_weight(Weight& w, const std::string& name, const std::vector<float>& host, int n_out, int n_in) {
    w.name = name; w.n_out = n_out; w.n_in = n_in;
    if ((size_t)n_out * n_in != host.size()) throw std::runtime_error("shape mismatch for " + name);
    const int at = act_type();
    if (at == OUT_F32) { upload(w.data, host); return; }
    DevBuf tmp; upload(tmp, host);
    w.data.alloc(host.size() * 2, false);
    convert_to(tmp.as<float>(), w.data.p, host.size(), at, st_);
    NSB_CUDA(cudaStreamSynchronize(st_));
}

// Q8_0 block = fp16 d + 32 x int8 along ne0 (scripts/convert_to_gguf.py:93-129). Split into planes; tensors of another type are
// quantised here with the converter's rule (d = amax / 127 stored as fp16, q = round(x / fp16(d))).
static void q8_planes(const GgufFile& g, const std::string& name, std::vector<int8_t>& q, std::vector<uint16_t>& d) {
    const GgufTensor& t = g.require(name);
    const size_t n = (size_t)t.n_elements(), nb = n / 32;
    const size_t q0 = q.size(), d0 = d.size();
    q.resize(q0 + n); d.resize(d0 + nb);
    if (t.type == GGML_Q8_0) {
        const std::vector<uint8_t> raw = g.read(t);
        for (size_t b = 0; b < nb; ++b) { memcpy(&d[d0 + b], &raw[b * 34], 2); memcpy(&q[q0 + b * 32], &raw[b * 34 + 2], 32); }
        return;
    }
    const std::vector<float> x = read_matrix_f32(g, name);
    for (size_t b = 0; b < nb; ++b) {
        float amax = 0.f; for (int i = 0; i < 32; ++i) amax = std::max(amax, std::fabs(x[b * 32 + i]));
        const __half dh = __float2half_rn(amax / 127.0f); uint16_t bits; memcpy(&bits, &dh, 2); d[d0 + b] = bits;
        const float df = __half2float(dh);
        for (int i = 0; i < 32; ++i) q[q0 + b * 32 + i] = (int8_t)(df > 0.f ? std::nearbyint(x[b * 32 + i] / df) : 0.f);
    }
}

// Chunked asynchronous host -> device copy out of the mapped file: the bytes go mmap -> one of two pinned chunks -> cudaMemcpyAsync on
// the engine stream; while chunk i is in flight the host fills chunk i + 1. Returns once everything is ENQUEUED (src is no longer
// read); consumers are ordered behind it on the same stream.
void Engine::stream_upload(void* dst, const uint8_t* src, size_t bytes) {
    constexpr size_t CHUNK = 16u << 20;
    if (!up_[0].p) for (int i = 0; i < 2; ++i) { up_[i].alloc(CHUNK); NSB_CUDA(cudaEventCreateWithFlags(&up_ev_[i], cudaEventDisableTiming)); }
    for (size_t off = 0; off < bytes; off += CHUNK) {
        const size_t n = std::min(CHUNK, bytes - off);
        NSB_CUDA(cudaEventSynchronize(up_ev_[up_k_]));              // the copy that last used this chunk has finished
        memcpy(up_[up_k_].p, src + off, n);
        NSB_CUDA(cudaMemcpyAsync((char*)dst + off, up_[up_k_].p, n, cudaMemcpyHostToDevice, st_));
        NSB_CUDA(cudaEventRecord(up_ev_[up_k_], st_));
        up_k_ ^= 1;
    }
}

void Engine::load_layer_matrix(Weight& w, const GgufFile& g, const std::string& out_name, const std::vector<std::string>& parts, int n_out, int n_in) {
    w.name = out_name; w.n_out = n_out; w.n_in = n_in;
    if (n_out % (int)parts.size() != 0 || n_in % 64 != 0) throw std::runtime_error("shape mismatch for " + out_name);
    const size_t rows = (size_t)n_out / parts.size(), part_elems = rows * n_in;
    // tensor-type / shape validation with the tensor's name in the message (the reference's loader only checks presence, nemo-ggml.cpp:362-384)
    for (const std::string& pn : parts) {
        const GgufTensor& t = g.require(pn);
        const bool squeezed3d = t.ne.size() == 3 && t.ne[0] == 1 && t.ne[1] == n_in;        // pointwise conv kept as (out, in, 1) by an older converter
        if ((size_t)t.n_elements() != part_elems || !(t.ne.size() >= 2 && (t.ne[0] == n_in || squeezed3d))) {
            std::string dims; for (auto d : t.ne) dims += (dims.empty() ? "" : ", ") + std::to_string(d);
            throw std::runtime_error("gguf: tensor '" + pn + "' has shape [" + dims + "], expected [" + std::to_string(n_in) + ", " + std::to_string(rows) + "] (ne0 = input features)");
        }
        if (t.type != GGML_F32 && t.type != GGML_F16 && t.type != GGML_Q8_0 && t.type != GGML_Q4_0)
            throw std::runtime_error("gguf: tensor '" + pn + "' has type " + std::to_string(t.type) + "; per-layer matrices must be F32, F16, Q8_0 or Q4_0");
    }
    if (d_raw_.bytes < part_elems * 4) { NSB_CUDA(cudaStreamSynchronize(st_)); d_raw_.alloc((size_t)D_FF * D_MODEL * 4, false); }
    if (q8_planes_mode()) {
        // Q4_0 files keep their nibbles in HBM in the fast mode (0.5625 bytes per weight; the fused kernel's Q4 variant); the strict
        // mode widens them to int8 quants q - 8 once (its integer block dots take any int8 weight)
        bool all_q4 = true;
        for (const std::string& pn : parts) all_q4 = all_q4 && g.require(pn).type == GGML_Q4_0;
        const bool nib = all_q4 && compute == NSB_COMPUTE_Q8_0;
        w.q4 = nib ? 1 : 0;
        w.data.alloc(nib ? (size_t)n_out * n_in / 2 : (size_t)n_out * n_in, false); w.scales.alloc((size_t)n_out * (n_in / 32) * 2, false);
        for (size_t i = 0; i < parts.size(); ++i) {
            const GgufTensor& t = g.require(parts[i]);
            uint16_t* dd = w.scales.as<uint16_t>() + i * (part_elems / 32);
            if (t.type == GGML_Q8_0) {                              // stays quantised: raw blocks up, split into planes on the device
                stream_upload(d_raw_.p, g.data(t), t.nbytes);
                unpack_q8_planes_kernel<<<grid_for(part_elems / 32), 256, 0, st_>>>(d_raw_.as<uint16_t>(), w.data.as<int8_t>() + i * part_elems, dd, part_elems / 32);
            } else if (all_q4) {
                stream_upload(d_raw_.p, g.data(t), t.nbytes);
                unpack_q4_planes_kernel<<<grid_for(part_elems / 32), 256, 0, st_>>>(d_raw_.as<uint16_t>(), w.data.as<uint8_t>() + i * (nib ? part_elems / 2 : part_elems), dd,
                                                                                   part_elems / 32, nib ? 0 : 1);
            } else {                                                // another stored type: quantised here with the converter's rule (host)
                std::vector<int8_t> q; std::vector<uint16_t> d; q8_planes(g, parts[i], q, d);
                NSB_CUDA(cudaStreamSynchronize(st_));
                h2d_sync(w.data.as<int8_t>() + i * part_elems, q.data(), q.size()); h2d_sync(dd, d.data(), d.size() * 2);
            }
        }
        return;
    }
    const int at = act_type();
    const size_t es = act_size();
    w.data.alloc((size_t)n_out * n_in * es, false);
    for (size_t i = 0; i < parts.size(); ++i) {
        const GgufTensor& t = g.require(parts[i]);
        void* dst = (char*)w.data.p + i * part_elems * es;
        const bool direct = (t.type == GGML_F32 && at == OUT_F32) || (t.type == GGML_F16 && at == OUT_F16);
        stream_upload(direct ? dst : d_raw_.p, g.data(t), t.nbytes);
        if (direct) continue;
        if (t.type == GGML_F32) convert_kernel<<<grid_for(part_elems), 256, 0, st_>>>(d_raw_.as<float>(), dst, part_elems, at);
        else if (t.type == GGML_F16) cvt_f16_kernel<<<grid_for(part_elems), 256, 0, st_>>>(d_raw_.as<__half>(), dst, part_elems, at);
        else dequant_blocks_kernel<<<grid_for(part_elems / 32), 256, 0, st_>>>(d_raw_.as<uint16_t>(), dst, part_elems / 32, t.type == GGML_Q4_0 ? 1 : 0, at);
    }
}

void Engine::load_weights(const GgufFile& g) {
    auto vec = [&](DevBuf& d, const std::string& n, size_t expect) {
        std::vector<float> h = g.read_f32(n);
        if (h.size() != expect) throw std::runtime_error("unexpected size for " + n);
        upload(d, h);
    };
    // matrices every GGUF keeps in F32: fp32 SIMT in strict mode; on the tensor cores (16-bit / Q8_0 modes) as 3xTF32 -- the
    // split copy [hi | lo | hi] goes to `scales` (NSB_STEM_TF32=1: single-pass tf32 on the plain copy, for A/B measurements)
    auto f32_weight = [&](Weight& w, const std::string& n, int n_out, int n_in, std::vector<float> h) {
        w.name = n; w.n_out = n_out; w.n_in = n_in; w.f32 = true; upload(w.data, h);
        if (!strict() && tf32x3_enabled()) upload(w.scales, tf32x3_weight(h, n_out, n_in));
        named_[n] = &w;
    };
    // ---- front-end tables (src/preprocessor.cpp:80-110, :296-299) ----
    {
        std::vector<float> win = g.read_f32("preprocessor.featurizer.window"), fb = g.read_f32("preprocessor.featurizer.fb");
        if (win.size() != WIN || fb.size() != (size_t)N_MELS * N_BINS) throw std::runtime_error("preprocessor tensor sizes");
        std::vector<float> w512(N_FFT, 0.f), c(N_FFT), s(N_FFT), fbt((size_t)N_BINS * N_MELS);
        memcpy(w512.data() + (N_FFT - WIN) / 2, win.data(), WIN * sizeof(float));
        for (int i = 0; i < N_FFT; ++i) { const float th = (2.0f * (float)M_PI * i) / N_FFT; s[i] = sinf(th); c[i] = cosf(th); }
        for (int m = 0; m < N_MELS; ++m) for (int k = 0; k < N_BINS; ++k) fbt[(size_t)k * N_MELS + m] = fb[(size_t)m * N_BINS + k];
        // [257][128] transposed weights, then per mel bin the span [lo, hi) of its non-zero weights (2 x 128 ints)
        fbt.resize((size_t)N_BINS * N_MELS + 2 * N_MELS);
        for (int m = 0; m < N_MELS; ++m) {
            int lo = N_BINS, hi = 0;
            for (int k = 0; k < N_BINS; ++k) if (fb[(size_t)m * N_BINS + k] != 0.0f) { lo = std::min(lo, k); hi = k + 1; }
            if (hi == 0) lo = 0;
            memcpy(&fbt[(size_t)N_BINS * N_MELS + m], &lo, 4); memcpy(&fbt[(size_t)N_BINS * N_MELS + N_MELS + m], &hi, 4);
        }
        upload(window_, w512); upload(cos_t_, c); upload(sin_t_, s); upload(fb_t_, fbt);
    }
    // ---- subsampling stem: always f32 (never quantised by the converter, convert_to_gguf.py:226) ----
    {
        auto conv_t = [&](DevBuf& d, const std::string& n) {           // [256][1][3][3] -> tap-major [9][256]
            std::vector<float> w = g.read_f32(n), t((size_t)9 * SUB_CH);
            if (w.size() != (size_t)SUB_CH * 9) throw std::runtime_error("unexpected size for " + n);
            for (int oc = 0; oc < SUB_CH; ++oc) for (int k = 0; k < 9; ++k) t[(size_t)k * SUB_CH + oc] = w[(size_t)oc * 9 + k];
            upload(d, t);
        };
        const std::string p = "encoder.pre_encode.";
        conv_t(c0_w_, p + "conv.0.weight"); vec(c0_b_, p + "conv.0.bias", SUB_CH);
        conv_t(c2_w_, p + "conv.2.weight"); vec(c2_b_, p + "conv.2.bias", SUB_CH);
        conv_t(c5_w_, p + "conv.5.weight"); vec(c5_b_, p + "conv.5.bias", SUB_CH);
        f32_weight(c3_w_, p + "conv.3.weight", SUB_CH, SUB_CH, g.read_f32(p + "conv.3.weight")); vec(c3_b_, p + "conv.3.bias", SUB_CH);
        f32_weight(c6_w_, p + "conv.6.weight", SUB_CH, SUB_CH, g.read_f32(p + "conv.6.weight")); vec(c6_b_, p + "conv.6.bias", SUB_CH);
        // out linear: reference flattens (c*17 + w) (nemo-ggml.cpp:937-940); our activations are NHWC so permute columns to (w*256 + c)
        std::vector<float> w = g.read_f32(p + "out.weight"), wp(w.size());
        if (w.size() != (size_t)D_MODEL * SUB_CH * SUB_W) throw std::runtime_error("pre_encode.out.weight size");
        for (int n = 0; n < D_MODEL; ++n) for (int c = 0; c < SUB_CH; ++c) for (int x = 0; x < SUB_W; ++x)
            wp[(size_t)n * SUB_CH * SUB_W + x * SUB_CH + c] = w[(size_t)n * SUB_CH * SUB_W + c * SUB_W + x];
        f32_weight(sub_out_w_, p + "out.weight", D_MODEL, SUB_CH * SUB_W, std::move(wp));
        vec(out_b_, p + "out.bias", D_MODEL);
    }
    // ---- conformer layers ----
    layers_.resize(n_layers);
    for (int l = 0; l < n_layers; ++l) {
        LayerW& L = layers_[l];
        const std::string p = "encoder.layers." + std::to_string(l) + ".";
        const char* norms[5] = {"norm_feed_forward1", "norm_self_att", "norm_conv", "norm_feed_forward2", "norm_out"};
        for (int i = 0; i < 5; ++i) { vec(L.ln[2 * i], p + norms[i] + ".weight", D_MODEL); vec(L.ln[2 * i + 1], p + norms[i] + ".bias", D_MODEL); }
        auto mat = [&](Weight& w, const std::string& n, int n_out, int n_in) { load_layer_matrix(w, g, p + n, {p + n}, n_out, n_in); };
        mat(L.ff1a, "feed_forward1.linear1.weight", D_FF, D_MODEL);
        mat(L.ff1b, "feed_forward1.linear2.weight", D_MODEL, D_FF);
        mat(L.ff2a, "feed_forward2.linear1.weight", D_FF, D_MODEL);
        mat(L.ff2b, "feed_forward2.linear2.weight", D_MODEL, D_FF);
        // q | k | v stacked along the output dim -> one GEMM with N = 3072
        load_layer_matrix(L.qkv, g, p + "self_attn.linear_qkv.weight",
                          {p + "self_attn.linear_q.weight", p + "self_attn.linear_k.weight", p + "self_attn.linear_v.weight"}, 3 * D_MODEL, D_MODEL);
        mat(L.out, "self_attn.linear_out.weight", D_MODEL, D_MODEL);
        mat(L.pw1, "conv.pointwise_conv1.weight", 2 * D_MODEL, D_MODEL);
        mat(L.pw2, "conv.pointwise_conv2.weight", D_MODEL, D_MODEL);
        vec(L.bias_u, p + "self_attn.pos_bias_u", D_MODEL); vec(L.bias_v, p + "self_attn.pos_bias_v", D_MODEL);
        {
            const GgufTensor& dw = g.require(p + "conv.depthwise_conv.weight");       // ggml [1024, k]: tap-major
            if (dw.ne.size() != 2 || dw.ne[0] != D_MODEL || dw.ne[1] != CONV_K)
                throw std::runtime_error("depthwise conv weight must be [1024, 9] (2-D, tap-major; reconvert old 3-D files)");
            vec(L.dw_w, p + "conv.depthwise_conv.weight", (size_t)CONV_K * D_MODEL);
        }
        vec(L.cln_g, p + "conv.batch_norm.weight", D_MODEL); vec(L.cln_b, p + "conv.batch_norm.bias", D_MODEL);
        for (Weight* w : {&L.ff1a, &L.ff1b, &L.ff2a, &L.ff2b, &L.qkv, &L.out, &L.pw1, &L.pw2}) named_[w->name] = w;
        { int k = 0; for (Weight* w : {&L.ff1a, &L.ff1b, &L.qkv, &L.out, &L.pw1, &L.pw2, &L.ff2a, &L.ff2b}) w->shadow_slot = k++; }
    }
    // ---- decoder + joint: always f32 ----
    {
        const std::string d = "decoder.prediction.";
        vec(embed_, d + "embed.weight", (size_t)VOCAB * HID);
        for (int l = 0; l < 2; ++l) {
            vec(lstm_w_[2 * l], d + "dec_rnn.lstm.weight_ih_l" + std::to_string(l), (size_t)4 * HID * HID);
            vec(lstm_w_[2 * l + 1], d + "dec_rnn.lstm.weight_hh_l" + std::to_string(l), (size_t)4 * HID * HID);
            vec(lstm_b_[2 * l], d + "dec_rnn.lstm.bias_ih_l" + std::to_string(l), (size_t)4 * HID);
            vec(lstm_b_[2 * l + 1], d + "dec_rnn.lstm.bias_hh_l" + std::to_string(l), (size_t)4 * HID);
        }
        f32_weight(joint_enc_w_, "joint.enc.weight", JOINT, D_MODEL, g.read_f32("joint.enc.weight"));
        vec(joint_enc_b_, "joint.enc.bias", JOINT);
        vec(pred_w_, "joint.pred.weight", (size_t)JOINT * HID); vec(pred_b_, "joint.pred.bias", JOINT);
        vec(jout_w_, "joint.joint_net.2.weight", (size_t)VOCAB * JOINT); vec(jout_b_, "joint.joint_net.2.bias", VOCAB);
    }
}

int q8_dense_min_rows();
void Engine::alloc_state() {
    const int S = max_streams, Cap = ATT_L + T, M = PRE_CACHE + 8 * T;
    const int t1 = M / 2 + 1, t2 = t1 / 2 + 1, t3 = t2 / 2 + 1;
    if (t3 != T + DROP_PRE) throw std::runtime_error("unexpected subsampling length");
    // per-slot state: max_streams stream slots + ONE private slot (index max_streams) for the non-streaming batch path, which needs
    // conv / decoder state of its own whatever the streams are doing
    const size_t SS = (size_t)S + 1;
    kv_.alloc(SS * n_layers * 2 * Cap * D_MODEL * kv_elem_size(kv_dtype));               // zero-initialised (nemo-stream.cpp:292-297)
    conv_cache_.alloc(SS * 2 * n_layers * (CONV_K - 1) * D_MODEL * 4); cc_par_.alloc(SS * 4);
    mel_hist_.alloc(SS * PRE_CACHE * N_MELS * 4);                                         // 9 zero frames (:59-60)
    ring_pos_.alloc(SS * 4); valid_len_.alloc(SS * 4);
    dec_h_.alloc(SS * 4 * HID * 4); dec_c_.alloc(SS * 4 * HID * 4);                      // [S][2 parities][2 layers][640]
    dec_proj_.alloc(SS * JOINT * 4);
    prev_token_.alloc(SS * 4); cand_valid_.alloc(SS * 4); dec_par_.alloc(SS * 4);
    hs_.assign(S, HostStream());
    for (int s = 0; s <= S; ++s) zero_slot(s);

    rl_ = hs_row_len(T);                                                                  // 1280 T + 353 samples per stream-step
    const size_t Mrows = (size_t)S * T;
    ensure_q8s_scratch((int)std::max<size_t>(Mrows, ATT_L + 2 * T));
    for (StepIO& io : io_) io.d_pcm.alloc((size_t)S * rl_ * 2);
    d_slot_.alloc((size_t)S * 4);
    mel_new_.alloc((size_t)S * 8 * T * N_MELS * 4);
    const size_t sp = (!strict() && tf32x3_enabled()) ? 2 : 1;        // 3xTF32: stem activations as [hi | lo] pixels
    dw_.alloc(sp * S * t2 * 33 * SUB_CH * 4);
    pw_.alloc((size_t)S * t2 * 33 * SUB_CH * 4);
    if (sp == 2) a3_.alloc(std::max((size_t)S * t3 * SUB_W * SUB_CH, (size_t)S * T * D_MODEL) * 2 * 4, false);   // split A of the stem projection / joint.enc
    x_.alloc(Mrows * D_MODEL * 4);
    a_.alloc(Mrows * D_MODEL * act_size());
    big_.alloc(Mrows * D_FF * act_size());
    // small batches: the QKV / pointwise-1 GEMMs run split-K and leave their partial planes for the consumer kernel to sum
    const size_t planes = Mrows <= SPLIT_CONSUMER_MAX_ROWS ? 4 : 1;
    consumer_planes_ = (int)planes;
    if (compute == NSB_COMPUTE_Q8_0) wscratch_.alloc((size_t)D_FF * D_MODEL * 2, false);   // largest layer matrix as fp16 (q8_predequant: op_gemm / bench_gemm)
    if (compute == NSB_COMPUTE_Q8_0 && (int)Mrows >= q8_dense_min_rows()) {                // layer-ahead fp16 shadows (see engine.h)
        const size_t sz[8] = {(size_t)D_FF * D_MODEL, (size_t)D_MODEL * D_FF, (size_t)3 * D_MODEL * D_MODEL, (size_t)D_MODEL * D_MODEL,
                              (size_t)2 * D_MODEL * D_MODEL, (size_t)D_MODEL * D_MODEL, (size_t)D_FF * D_MODEL, (size_t)D_MODEL * D_FF};
        size_t off = 0; for (int k = 0; k < 8; ++k) { shadow_off_[k] = off; off += sz[k] * 2; }
        shadow_bytes_ = off;
        for (DevBuf& b : shadow_) b.alloc(off, false);
        NSB_CUDA(cudaStreamCreateWithFlags(&st_deq_, cudaStreamNonBlocking));
        ev_deq_.resize(n_layers); ev_lstart_.resize(n_layers + 1);
        for (cudaEvent_t& e : ev_deq_) NSB_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        for (cudaEvent_t& e : ev_lstart_) NSB_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    }
    qkv_.alloc(planes * Mrows * 3 * D_MODEL * 4);
    pw1_.alloc(planes * Mrows * 2 * D_MODEL * 4);
    encp_.alloc(Mrows * JOINT * 4);
    part_.alloc((size_t)MAX_SPLITS * std::min<size_t>(Mrows, 1024) * D_MODEL * 4);       // split-K workspace (only used when rows <= 1024)
    out_tok_.alloc((size_t)S * MAX_SYMBOLS * T * 4); out_cnt_.alloc((size_t)S * 4);
    dec_sync_.alloc(decode_sync_bytes(S));
    for (Side& sd : side_) {                                                             // hand-over buffers of a step, one set per step in flight (decode overlap)
        sd.slot.alloc((size_t)S * 4); sd.encp.alloc(Mrows * JOINT * 4); sd.out_tok.alloc((size_t)S * MAX_SYMBOLS * T * 4);
        sd.out_cnt.alloc((size_t)S * 4); sd.sync.alloc(decode_sync_bytes(S));
    }
    for (StepIO& io : io_) {
        io.h_pcm.alloc((size_t)S * rl_ * 2); io.h_slot.alloc((size_t)S * 4);
        io.h_tok.alloc((size_t)S * MAX_SYMBOLS * T * 4); io.h_cnt.alloc((size_t)S * 4);
    }
}

void Engine::zero_slot(int s) {
    NSB_CUDA(cudaSetDevice(device_));
    join_decode_stream();                                                      // decoder state of the slot: no decode may still be running
    const int Cap = ATT_L + T;
    const size_t kvb = (size_t)n_layers * 2 * Cap * D_MODEL * kv_elem_size(kv_dtype);
    NSB_CUDA(cudaMemsetAsync((char*)kv_.p + (size_t)s * kvb, 0, kvb, st_));
    const size_t cb = (size_t)2 * n_layers * (CONV_K - 1) * D_MODEL * 4;
    NSB_CUDA(cudaMemsetAsync((char*)conv_cache_.p + (size_t)s * cb, 0, cb, st_));
    NSB_CUDA(cudaMemsetAsync((char*)cc_par_.p + (size_t)s * 4, 0, 4, st_));
    NSB_CUDA(cudaMemsetAsync((char*)mel_hist_.p + (size_t)s * PRE_CACHE * N_MELS * 4, 0, (size_t)PRE_CACHE * N_MELS * 4, st_));
    NSB_CUDA(cudaMemsetAsync((char*)dec_h_.p + (size_t)s * 4 * HID * 4, 0, (size_t)4 * HID * 4, st_));
    NSB_CUDA(cudaMemsetAsync((char*)dec_c_.p + (size_t)s * 4 * HID * 4, 0, (size_t)4 * HID * 4, st_));
    NSB_CUDA(cudaMemsetAsync((char*)dec_par_.p + (size_t)s * 4, 0, 4, st_));
    const int zero = 0, blank = BLANK;
    NSB_CUDA(cudaMemcpyAsync((char*)ring_pos_.p + (size_t)s * 4, &zero, 4, cudaMemcpyHostToDevice, st_));
    NSB_CUDA(cudaMemcpyAsync((char*)valid_len_.p + (size_t)s * 4, &zero, 4, cudaMemcpyHostToDevice, st_));
    NSB_CUDA(cudaMemcpyAsync((char*)cand_valid_.p + (size_t)s * 4, &zero, 4, cudaMemcpyHostToDevice, st_));
    NSB_CUDA(cudaMemcpyAsync((char*)prev_token_.p + (size_t)s * 4, &blank, 4, cudaMemcpyHostToDevice, st_));   // prev_token = blank (:41-42)
    NSB_CUDA(cudaStreamSynchronize(st_));
    if (s < max_streams) hs_clear(hs_[s]);
}

// P_l = linear_pos(pos_emb rows) for the L+2T-1 relative positions a chunk can touch, once, at load.
// (The reference recomputes mul_mat(attn_pos_w, pos_emb) over 2K-1 rows per layer per chunk, nemo-stream.cpp:488.)
void Engine::build_pos_tables(const GgufFile& g) {
    const int n_rel = ATT_L + 2 * T - 1;
    std::vector<float> tab((size_t)n_rel * D_MODEL);
    for (int r = 0; r < n_rel; ++r) pos_emb_row(r - (T - 1), &tab[(size_t)r * D_MODEL]);
    DevBuf d_tab; upload(d_tab, tab);
    DevBuf d_a; const void* A = d_tab.p;
    if (act_type() != OUT_F32) { d_a.alloc(tab.size() * 2, false); convert_to(d_tab.as<float>(), d_a.p, tab.size(), act_type(), st_); A = d_a.p; }
    for (int l = 0; l < n_layers; ++l) {
        const std::string n = "encoder.layers." + std::to_string(l) + ".self_attn.linear_pos.weight";
        Weight wpos; load_layer_matrix(wpos, g, n, {n}, D_MODEL, D_MODEL);
        // kept in the K/V ring dtype: the attention kernel stages this head's rows in shared memory next to K and V
        layers_[l].pos_proj.alloc((size_t)n_rel * D_MODEL * kv_elem_size(kv_dtype), false);
        if (kv_dtype == 0) gemm(A, D_MODEL, wpos, n_rel, nullptr, layers_[l].pos_proj.p, D_MODEL, EPI_NONE, 1.f, OUT_F32);
        else {
            DevBuf tmp; tmp.alloc((size_t)n_rel * D_MODEL * 4, false);
            gemm(A, D_MODEL, wpos, n_rel, nullptr, tmp.p, D_MODEL, EPI_NONE, 1.f, OUT_F32);
            convert_to(tmp.as<float>(), layers_[l].pos_proj.p, (size_t)n_rel * D_MODEL, kv_dtype == 1 ? OUT_F16 : OUT_BF16, st_);
            NSB_CUDA(cudaStreamSynchronize(st_));
        }
        NSB_CUDA(cudaStreamSynchronize(st_));
    }
}

void Engine::gemm(const void* A, long long lda, const Weight& W, int M, const float* bias, void* C, long long ldc, int epi, float alpha,
                  int out_type) {
    GemmArgs a; a.A = A; a.lda = lda; a.M = M; a.bias = bias; a.C = C; a.ldc = ldc;
    a.epi = epi; a.alpha = alpha; a.out_type = out_type; a.pair = 1;
    gemm(a, W);
}

void Engine::gemm(GemmArgs& a, const Weight& W) {
    a.W = W.data.p; a.w_scales = W.scales.p; a.q4 = W.q4; a.N = W.n_out; a.K = W.n_in;
    ProfScope ps(this, PC_GEMM);
    if (cur_shadow_ && W.shadow_slot >= 0) { a.W = cur_shadow_ + shadow_off_[W.shadow_slot]; a.w_scales = nullptr; a.q4 = 0; }   // dequantised a layer ahead
    else q8_predequant(W, a.M, a);
    if (compute == NSB_COMPUTE_Q8_0_STRICT) { launch_gemm_q8_strict(a, q8s_scratch_.p, q8s_scratch_.bytes, st_); count_launch(); }
    else if (compute == NSB_COMPUTE_F32) launch_gemm_simt(a, st_);
    else launch_gemm_tc(a, act_type(), st_);
    count_launch();
}

void Engine::ensure_q8s_scratch(int rows) {
    if (compute != NSB_COMPUTE_Q8_0_STRICT) return;
    const size_t need = q8_strict_scratch_bytes(rows, D_FF);
    if (q8s_scratch_.bytes < need) { NSB_CUDA(cudaStreamSynchronize(st_)); q8s_scratch_.alloc(need, false); }
}

// GEMM on a matrix every GGUF keeps in F32 (stem 1x1 convs, stem projection, joint.enc). Strict mode: fp32 SIMT. Tensor-core
// modes: 3xTF32 -- W = [hi | lo | hi] (load time), A = [hi | lo] written by the producer kernel (a_presplit) or by a split pass
// into a3_; NSB_STEM_TF32=1 falls back to single-pass tf32 on the plain fp32 operands.
void Engine::gemm_f32w(GemmArgs& g, const Weight& W, bool a_presplit) {
    if (strict()) { launch_gemm_simt(g, st_); count_launch(); return; }
    if (W.scales.p) {
        const int K = W.n_in;
        if (!a_presplit) {
            if (g.lda != K || (size_t)g.M * 2 * K * 4 > a3_.bytes) throw std::runtime_error("gemm_f32w: split scratch too small / strided A");
            launch_split_tf32((const float*)g.A, a3_.as<float>(), (size_t)g.M, K, st_); count_launch();
            g.A = a3_.p;
        }
        g.lda = 2 * K; g.a_fold = K; g.K = 3 * K; g.W = W.scales.p;
    }
    launch_gemm_tc(g, OUT_F32, st_); count_launch();
}

// Q8_0 mode, batches of >= 4 row tiles: dequantise the matrix once into an fp16 scratch (L2-resident hand-over to the GEMM that
// follows) instead of once per m-tile inside the fused kernel. Small batches keep the fused operand path (weight streaming).
// token rows per step from which Q8_0 / Q4_0 matrices are expanded to fp16 before the GEMMs (layer-ahead shadows in the step, a scratch
// per launch for single operator calls) instead of inside every m-tile CTA of the fused kernel. Default 1 = always: measured per step,
// shadows vs fused, 1 stream x 160 ms 2.05 vs 2.30 ms, 64 streams 2.38 vs 2.49, 128 streams 3.18 vs 3.55, 24 streams x 1.12 s 3.3 vs 4.7,
// 64 streams x 560 ms 3.74 vs 4.35 (profiles/r02_notes.md): the expansion runs on its own stream under the previous layer and the GEMMs
// then are the fp16 ones. NSB_Q8_PREDEQUANT_ROWS=<rows> brings the fused operand path back below that many rows (no shadows: 122 MB less).
int q8_dense_min_rows() {
    const char* e = getenv("NSB_Q8_PREDEQUANT_ROWS");          // read per call (engine creation, graph capture): a test can switch it between engines
    return e ? atoi(e) : 1;
}
void Engine::q8_predequant(const Weight& W, int M, GemmArgs& a) {
    const int min_rows = q8_dense_min_rows();
    if (compute != NSB_COMPUTE_Q8_0 || !W.scales.p || M < min_rows) return;
    if (q8_pair256_enabled()) return;                              // large batches: the dequantisation is fused into the CTA-pair tiles (gemm_q8_pair256_kernel)
    const size_t bytes = (size_t)W.n_out * W.n_in * 2;
    if (wscratch_.bytes < bytes) throw std::runtime_error("q8_predequant: scratch not allocated");   // sized in alloc_state (no allocation inside a graph capture)
    launch_dequant_q8(W.data.p, W.scales.p, wscratch_.p, W.n_out, W.n_in, st_, W.q4);
    count_launch();
    a.W = wscratch_.p; a.w_scales = nullptr; a.w_dynamic = 1; a.pair = 0; a.q4 = 0;
}

bool Engine::shadow_mode(int rows) const {
    static const bool off = [] { const char* e = getenv("NSB_Q8_SHADOW"); return e && e[0] == '0'; }();
    const int min_rows = q8_dense_min_rows();
    return !off && !q8_pair256_enabled() && compute == NSB_COMPUTE_Q8_0 && shadow_bytes_ && rows >= min_rows && !profiling_;
}
// all 8 matrices of layer l -> fp16 in shadow_[l % 2], on stream s (same fp16(d) * q values as the fused operand path)
void Engine::dequant_layer_async(int l, cudaStream_t s) {
    LayerW& L = layers_[l];
    char* base = shadow_[l & 1].as<char>();
    for (Weight* w : {&L.ff1a, &L.ff1b, &L.qkv, &L.out, &L.pw1, &L.pw2, &L.ff2a, &L.ff2b}) {
        launch_dequant_q8(w->data.p, w->scales.p, base + shadow_off_[w->shadow_slot], w->n_out, w->n_in, s, w->q4);
        count_launch();
    }
}

bool Engine::split_consumers(int rows) const {
    static const bool off = [] { const char* e = getenv("NSB_NO_SPLIT_CONSUMERS"); return e && e[0] == '1'; }();
    return !off && !pair_gemm_enabled() && consumer_planes_ >= 4 && (compute == NSB_COMPUTE_F16 || compute == NSB_COMPUTE_BF16) && rows <= 128;
}

// split-K GEMM whose fp32 partial planes C[z][M][N] are left for the consumer kernel to sum (QKV -> attention, pointwise-1 -> conv module)
void Engine::gemm_planes(const void* A, long long lda, const Weight& W, int M, void* C, int planes) {
    GemmArgs a; a.A = A; a.lda = lda; a.W = W.data.p; a.w_scales = W.scales.p; a.q4 = W.q4; a.M = M; a.N = W.n_out; a.K = W.n_in; a.C = C; a.ldc = W.n_out;
    a.epi = EPI_PARTIAL; a.out_type = OUT_F32; a.splits = planes; a.force_bn = 64; a.force_stages = 4;
    { ProfScope ps(this, PC_GEMM); launch_gemm_tc(a, act_type(), st_); }
    count_launch();
}

void Engine::gemm_residual(const void* A, long long lda, const Weight& W, int M, float* x, float alpha) {
    // The N = 1024 GEMMs have few output tiles: with <= 1024 token rows the K dimension is split across CTAs so that
    // >= ~1 wave of SMs pulls weights; the fp32 partials land in part_ and the NEXT LayerNorm kernel adds them to x.
    int splits = 1;
    if (!strict() && M <= 1024) {
        const int tiles = ((M + 127) / 128) * (W.n_out / (W.n_in >= 4096 ? 64 : 32));
        const int nk = W.n_in / 64;
        while (splits < MAX_SPLITS && tiles * splits < 120 && nk % (splits * 2) == 0 && nk / (splits * 2) >= 2) splits *= 2;
    }
    // Large batches, K = 4096 (FFN down-projections): with 7 x 8 tiles the N = 1024 GEMM cannot fill the machine. Two K slices on 256 x 112
    // pair tiles = 7 x 10 x 2 = 140 tiles for the 148 co-resident pair slots; measured at 1792 rows (profiles/r02_gemm_sweep.txt):
    // 15.2 us (987 TFLOP/s) against 17.4 us for four slices of 256 x 256 tiles and 21.6 us unsplit. NSB_FFDOWN_SPLIT=1: off.
    static const int big_split = [] { const char* e = getenv("NSB_FFDOWN_SPLIT"); return e ? atoi(e) : 2; }();
    if (!strict() && M > 1024 && W.n_in >= 4096 && big_split > 1 && (size_t)big_split * M * D_MODEL * 4 <= part_.bytes) splits = big_split;
    if (splits == 1) { gemm(A, lda, W, M, nullptr, x, D_MODEL, EPI_RESID, alpha, OUT_F32); return; }
    GemmArgs a; a.A = A; a.lda = lda; a.W = W.data.p; a.w_scales = W.scales.p; a.q4 = W.q4; a.M = M; a.N = W.n_out; a.K = W.n_in; a.C = part_.p; a.ldc = D_MODEL;
    a.epi = EPI_PARTIAL; a.out_type = OUT_F32; a.splits = splits;
    { ProfScope ps(this, PC_GEMM);
      if (cur_shadow_ && W.shadow_slot >= 0) { a.W = cur_shadow_ + shadow_off_[W.shadow_slot]; a.w_scales = nullptr; } else q8_predequant(W, M, a);
      launch_gemm_tc(a, act_type(), st_); }
    count_launch();
    pending_.part = part_.as<float>(); pending_.n = splits; pending_.alpha = alpha;
}

// ------------------------------------------------------------------------------------------
// streams (host bookkeeping only; all arithmetic is on the device)
// ------------------------------------------------------------------------------------------
int Engine::open_stream() {
    collect_all();
    for (int s = 0; s < max_streams; ++s)
        if (!hs_[s].open) { zero_slot(s); hs_[s].open = true; return s; }
    throw std::runtime_error("no free stream slot (max_streams = " + std::to_string(max_streams) + ")");
}
void Engine::close_stream(int s) { collect_all(); if (s < 0 || s >= max_streams || !hs_[s].open) throw std::invalid_argument("bad stream id"); hs_release_pcm(hs_[s]); hs_[s].open = false; }
void Engine::reset_stream(int s) { collect_all(); if (s < 0 || s >= max_streams || !hs_[s].open) throw std::invalid_argument("bad stream id"); zero_slot(s); }

void Engine::push_pcm(int s, const int16_t* pcm, int n) {
    if (s < 0 || s >= max_streams || !hs_[s].open) throw std::invalid_argument("bad stream id");
    if (!pcm || n <= 0) return;                                        // reference returns "" on null/<=0 (nemo-stream.cpp:1079)
    hs_push(hs_[s], pcm, n);
}

// chunk gate and PCM row of a stream: host_stream.h (pure host code, driven on CPU by tests/test_host_api.py)
bool Engine::ready(int s) const { return hs_ready(hs_[s], T); }

// Up to MAX_INFLIGHT (three) steps in flight: step i+1 is staged and enqueued while step i runs, so the device never waits for the
// host between steps; the third slot lets the encoder of step i+2 be queued before the decode of step i has finished (decode overlap:
// a step with many symbol rounds decodes longer than one encoder pass; with two slots the engine stream then idled until the host
// came back from step_end). Host buffers (pinned PCM rows, slots, token ids) and the device-side hand-over buffers are rings of that
// depth; the device-side step workspace is shared -- everything is ordered on the engine stream.
int Engine::step_begin() {
    if (n_inflight_ == MAX_INFLIGHT) throw std::runtime_error("step_begin: three steps are already in flight (call step_end)");
    NSB_CUDA(cudaSetDevice(device_));
    std::vector<int> batch;
    for (int s = 0; s < max_streams; ++s) if (ready(s)) batch.push_back(s);
    const int B = (int)batch.size();
    if (!B) return 0;
    StepIO& io = io_[io_next_];
    int16_t* hp = io.h_pcm.as<int16_t>(); int* hsl = io.h_slot.as<int>();
    for (int b = 0; b < B; ++b) {
        HostStream& h = hs_[batch[b]];
        hs_stage_row(h, T, rl_, hp + (size_t)b * rl_); hsl[b] = batch[b];
        hs_launched(h, T);                                                // ready() now asks for the NEXT chunk; samples no later chunk needs are dropped
    }
    const int side = side_acquire();
    // PCM rows go up on the copy stream (4.8 MB per step at 256 streams x 560 ms: 0.2 ms that used to sit between two steps' kernels on the
    // engine stream); the buffer belongs to this step's slot of the in-flight ring, whose previous user was collected by step_end
    NSB_CUDA(cudaMemcpyAsync(io.d_pcm.p, hp, (size_t)B * rl_ * 2, cudaMemcpyHostToDevice, st_copy_));
    NSB_CUDA(cudaEventRecord(io.h2d, st_copy_));
    NSB_CUDA(cudaStreamWaitEvent(st_, io.h2d, 0));
    NSB_CUDA(cudaMemcpyAsync(side_[side].slot.p, hsl, (size_t)B * 4, cudaMemcpyHostToDevice, st_));
    NSB_CUDA(cudaEventRecord(io.ev0, st_));
    // the decode's stream: its tokens go home behind it. A step begun while another one is in flight is part of a pipeline
    cudaStream_t tail = run_step(B, io.d_pcm.as<int16_t>(), side, n_inflight_ >= 1);
    NSB_CUDA(cudaEventRecord(io.ev1, tail));
    NSB_CUDA(cudaMemcpyAsync(io.h_cnt.p, side_[side].out_cnt.p, (size_t)B * 4, cudaMemcpyDeviceToHost, tail));
    NSB_CUDA(cudaMemcpyAsync(io.h_tok.p, side_[side].out_tok.p, (size_t)B * MAX_SYMBOLS * T * 4, cudaMemcpyDeviceToHost, tail));
    NSB_CUDA(cudaEventRecord(io.done, tail));
    if (tail != st_) { NSB_CUDA(cudaEventRecord(side_[side].dec_done, tail)); }   // the side is free again once its tokens have left
    io.batch = std::move(batch);
    io_next_ = (io_next_ + 1) % MAX_INFLIGHT; n_inflight_ += 1;
    return B;
}

int Engine::step_end() {
    if (n_inflight_ == 0) return 0;
    NSB_CUDA(cudaSetDevice(device_));
    StepIO& io = io_[(io_next_ + MAX_INFLIGHT - n_inflight_) % MAX_INFLIGHT];   // the OLDEST step in flight
    n_inflight_ -= 1;
    const int B = (int)io.batch.size();
    NSB_CUDA(cudaEventSynchronize(io.done));
    float ms = 0.f; NSB_CUDA(cudaEventElapsedTime(&ms, io.ev0, io.ev1));
    stats.steps += 1; stats.chunks += B; stats.device_ms += ms; stats.last_step_ms = ms;
    collect_tokens(io);
    io.batch.clear();
    return B;
}

void Engine::collect_all() { while (n_inflight_) step_end(); }

int Engine::step() {
    collect_all();
    const int B = step_begin();
    if (B) step_end();
    return B;
}

void Engine::collect_tokens(StepIO& io) {
    const int* cnt = io.h_cnt.as<int>(); const int* tok = io.h_tok.as<int>();
    const int B = (int)io.batch.size();
    for (int b = 0; b < B; ++b) {
        HostStream& h = hs_[io.batch[b]];
        for (int i = 0; i < cnt[b] && i < MAX_SYMBOLS * T; ++i) h.tokens.push_back(tok[(size_t)b * MAX_SYMBOLS * T + i]);
        h.chunks_done += 1;
    }
}

int Engine::pop_tokens(int s, int32_t* out, int cap) {
    if (s < 0 || s >= max_streams) throw std::invalid_argument("bad stream id");
    HostStream& h = hs_[s]; int n = 0;
    while (n < cap && !h.tokens.empty()) { out[n++] = h.tokens.front(); h.tokens.pop_front(); }
    return n;
}
int Engine::chunks(int s) const { if (s < 0 || s >= max_streams) throw std::invalid_argument("bad stream id"); return (int)hs_[s].chunks_done; }

// tokens_to_text (src/nemo-ggml.cpp:1432-1458, timestamps off): piece starting with U+2581 -> ' ' + rest
std::string Engine::detok(const int32_t* t, int n) const {
    std::string r;
    for (int i = 0; i < n; ++i) {
        const int id = t[i];
        if (id < 0 || id >= VOCAB) continue;
        char piece[9]; memcpy(piece, &vocab[(size_t)id * 8], 8); piece[8] = 0;
        const std::string pc(piece);
        if (pc.size() >= 3 && strncmp(pc.c_str(), "\xe2\x96\x81", 3) == 0) { r += ' '; r += pc.substr(3); } else r += pc;
    }
    return r;
}

// Diagnostic only (NSB_SKIP=ln,attn,conv,decode,ff,qkv,out,pw,sub,mel): leave kernel classes out of the step to read their
// in-graph marginal cost off the step time. Results are meaningless with anything skipped.
static unsigned skip_mask() {
    static const unsigned m = [] {
        unsigned v = 0; const char* e = getenv("NSB_SKIP"); if (!e) return v;
        const char* names[] = {"ln", "attn", "conv", "decode", "ff", "qkv", "out", "pw", "sub", "mel"};
        for (int i = 0; i < 10; ++i) if (strstr(e, names[i])) v |= 1u << i;
        return v;
    }();
    return m;
}
enum { SK_LN = 1, SK_ATTN = 2, SK_CONV = 4, SK_DECODE = 8, SK_FF = 16, SK_QKV = 32, SK_OUT = 64, SK_PW = 128, SK_SUB = 256, SK_MEL = 512 };

// Decode overlap (nsb_engine_config::decode_overlap: 0 automatic, 1 always, 2 never; NSB_DECODE_OVERLAP=0/1 overrides): for batches of
// <= 512 token rows (NSB_DECODE_OVERLAP_ROWS). Up to 128 rows every encoder kernel launches <= 128 CTAs on the 148 SMs, so the 20 CTAs of
// the narrow decode cost the encoder nothing; up to ~512 rows the encoder loses less to them than the decode's latency-bound rounds
// take inline (measured per step: 224 rows 2.95 -> 2.57 ms, 448 rows 3.73 -> 3.28; at 896 rows 5.08 -> 5.84 and at 1792 rows 6.80 -> 8.78:
// off there). Automatic = only for steps that are part of a pipeline (a step begun while another is in flight, back-to-back bench steps):
// the narrow decode takes ~2x longer than the full-width one, which only pays when it hides under the next step's encoder. Off while
// taps / per-launch profiling are on (they read decode-side buffers behind a sync of st_ only) and in the strict modes.
bool Engine::overlap_decode(int rows, bool pipelined) const {
    static const int env = [] { const char* e = getenv("NSB_DECODE_OVERLAP"); return e ? atoi(e) : -1; }();
    const int mode = env == 0 ? 2 : env == 1 ? 1 : cfg_.decode_overlap;
    if (debug_ || profiling_ || strict() || mode == 2) return false;
    static const int max_rows = [] { const char* e = getenv("NSB_DECODE_OVERLAP_ROWS"); return e ? atoi(e) : 512; }();
    return mode == 1 || (rows <= max_rows && pipelined);
}

void Engine::join_decode_stream() {
    for (Side& q : side_) if (q.dec_pending) { NSB_CUDA(cudaStreamWaitEvent(st_, q.dec_done, 0)); q.dec_pending = false; }
}

int Engine::side_acquire() {
    const int p = side_next_;
    if (side_[p].dec_pending) { NSB_CUDA(cudaStreamWaitEvent(st_, side_[p].dec_done, 0)); side_[p].dec_pending = false; }
    return p;
}

template <class Key, class Fn>
void Engine::run_graphed(std::map<Key, StepGraph>& cache, const Key& key, cudaStream_t s, Fn&& body) {
    if (!cfg_.use_cuda_graph || debug_ || profiling_) { body(); return; }
    // bounded cache: a step graph exists per (batch size, staging buffer, side); serving with ever-changing batch sizes would otherwise
    // accumulate up to 4 x max_streams executables. Past the bound everything is dropped and re-captured on demand (both streams drained
    // first: an executable must not be destroyed under a launch that is still running).
    constexpr size_t MAX_GRAPHS = 96;
    if (cache.size() >= MAX_GRAPHS && cache.find(key) == cache.end()) {
        NSB_CUDA(cudaStreamSynchronize(st_)); NSB_CUDA(cudaStreamSynchronize(st_dec_));
        for (auto& e : cache) if (e.second.exec) cudaGraphExecDestroy(e.second.exec);
        cache.clear();
    }
    StepGraph& g = cache[key];
    if (!g.exec) {
        const long long before = stats.kernel_launches;
        cudaGraph_t graph = nullptr;
        NSB_CUDA(cudaStreamBeginCapture(s, cudaStreamCaptureModeRelaxed));
        try { body(); }
        catch (...) { cudaStreamEndCapture(s, &graph); if (graph) cudaGraphDestroy(graph); cache.erase(key); throw; }
        NSB_CUDA(cudaStreamEndCapture(s, &graph));
        const cudaError_t err = cudaGraphInstantiate(&g.exec, graph, 0);
        cudaGraphDestroy(graph);
        if (err != cudaSuccess) { cache.erase(key); throw CudaError(std::string("cudaGraphInstantiate: ") + cudaGetErrorString(err)); }
        g.launches = stats.kernel_launches - before;
        stats.kernel_launches = before;                                         // capture launched nothing yet
    }
    NSB_CUDA(cudaGraphLaunch(g.exec, s));
    stats.kernel_launches += g.launches;
}

cudaStream_t Engine::run_step(int B, const int16_t* d_pcm, int side, bool pipelined) {
    last_B_ = B;
    const bool ov = overlap_decode(B * T, pipelined);
    Side& sd = side_[side];
    if (!ov) join_decode_stream();                                              // decode on st_: behind any decode still running on the other stream
    run_graphed(graphs_, std::make_tuple(B, (const void*)d_pcm, side), st_, [&] { run_encoder_kernels(B, d_pcm, side); });
    if (ov) {
        NSB_CUDA(cudaEventRecord(sd.enc_done, st_));
        NSB_CUDA(cudaStreamWaitEvent(st_dec_, sd.enc_done, 0));
    }
    cudaStream_t s = ov ? st_dec_ : st_;
    if (!(skip_mask() & 8u /* SK_DECODE */))
        run_graphed(dec_graphs_, std::make_tuple(B, side, ov ? 1 : 0), s, [&] { run_decode_kernels(B, side, s, ov); });
    if (ov) { NSB_CUDA(cudaEventRecord(sd.dec_done, st_dec_)); sd.dec_pending = true; }
    side_next_ = (side + 1) % MAX_INFLIGHT;
    return s;
}

// ------------------------------------------------------------------------------------------
// THE HOT PATH: one batched chunk for B streams, PCM already in HBM, tokens left in HBM.
// ------------------------------------------------------------------------------------------
void Engine::run_encoder_kernels(int B, const int16_t* d_pcm, int side) {
    const unsigned skip = skip_mask();
    cur_shadow_ = nullptr;
    const int M = PRE_CACHE + 8 * T, t1 = M / 2 + 1, t2 = t1 / 2 + 1, t3 = t2 / 2 + 1;
    const int rows = B * T, at = act_type();
    const int* slot = side_[side].slot.as<int>();
    float* x = x_.as<float>();
    pending_ = PartialSum{};

    // P: log-mel of the 8T new frames per stream
    if (!(skip & SK_MEL)) { ProfScope ps(this, PC_MEL);
    launch_logmel(d_pcm, rl_, B, 8 * T, window_.as<float>(), cos_t_.as<float>(), sin_t_.as<float>(), fb_t_.as<float>(),
                  mel_new_.as<float>(), (size_t)8 * T * N_MELS, st_); }
    count_launch();
    if (debug_) { launch_mel_gather(mel_hist_.as<float>(), mel_new_.as<float>(), slot, B, T, dbg_mel_.as<float>(), st_); count_launch(); }
    // S: subsampling stem (NHWC)
    const bool tc = !strict();
    const int split = tc && c3_w_.scales.p ? 1 : 0;                    // stem producers write [hi | lo] pixels for the 3xTF32 GEMMs
    if (!(skip & SK_SUB)) { ProfScope ps(this, PC_SUBSAMPLE);
    launch_stem_conv0_dw(mel_hist_.as<float>(), mel_new_.as<float>(), slot, B, T, c0_w_.as<float>(), c0_b_.as<float>(), c2_w_.as<float>(),
                         c2_b_.as<float>(), dw_.as<float>(), st_, split);
    launch_mel_hist_update(mel_hist_.as<float>(), mel_new_.as<float>(), slot, B, T, st_);
    count_launch(2);
    // 1x1 convs + out projection: fp32 SIMT in strict-f32 mode, 3xTF32 on tcgen05 otherwise (these matrices are F32 in every GGUF)
    {
        GemmArgs g; g.A = dw_.p; g.lda = SUB_CH; g.W = c3_w_.data.p; g.M = B * t2 * 33; g.N = SUB_CH; g.K = SUB_CH; g.bias = c3_b_.as<float>();
        g.C = pw_.p; g.ldc = SUB_CH; g.epi = EPI_RELU; gemm_f32w(g, c3_w_, split);
    }
    launch_dwconv_s2(pw_.as<float>(), B, t2, 33, c5_w_.as<float>(), c5_b_.as<float>(), dw_.as<float>(), st_, split); count_launch();
    {
        GemmArgs g; g.A = dw_.p; g.lda = SUB_CH; g.W = c6_w_.data.p; g.M = B * t3 * SUB_W; g.N = SUB_CH; g.K = SUB_CH; g.bias = c6_b_.as<float>();
        g.C = pw_.p; g.ldc = SUB_CH; g.epi = EPI_RELU; gemm_f32w(g, c6_w_, split);
    }
    {   // flatten + out linear on the T kept frames (frames 0,1 of every stream are dropped: nemo-stream.cpp:136-144)
        GemmArgs g; g.W = sub_out_w_.data.p; g.N = D_MODEL; g.K = SUB_W * SUB_CH; g.bias = out_b_.as<float>(); g.ldc = D_MODEL; g.lda = SUB_W * SUB_CH;
        g.A = pw_.p;
        if (!tc) {                                                     // SIMT: gather only the kept rows
            g.group = T; g.group_stride = (long long)t3 * SUB_W * SUB_CH; g.row_off = DROP_PRE; g.M = rows; g.C = x; g.epi = EPI_NONE;
        } else {                                                       // tensor cores: all T+2 frames, dropped rows skipped by the epilogue row map
            g.M = B * t3; g.c_group = t3; g.c_drop = DROP_PRE;
            constexpr int SUB_SPLITS = 8;                              // K = 4352 = 136 k-blocks of 32 (x3 as 3xTF32); small batches need split-K to fill the SMs
            if (rows <= 1024 && (size_t)(SUB_SPLITS - 1) * rows * D_MODEL * 4 <= part_.bytes) {
                g.splits = SUB_SPLITS; g.epi = EPI_PARTIAL; g.C0 = x; g.C = part_.p;
                pending_.part = part_.as<float>(); pending_.n = SUB_SPLITS - 1; pending_.alpha = 1.f;   // summed by the first LayerNorm
            } else { g.C = x; g.epi = EPI_NONE; }
        }
        gemm_f32w(g, sub_out_w_, false);
    }
    }   // PC_SUBSAMPLE

    // L: cache-aware conformer layers
    const long long kv_slot_stride = (long long)n_layers * 2 * (ATT_L + T) * D_MODEL;
    const long long cc_par_stride = (long long)n_layers * (CONV_K - 1) * D_MODEL, cc_slot_stride = 2 * cc_par_stride;
    auto ln = [&](const float* g_, const float* b_) {
        if (skip & SK_LN) { pending_ = PartialSum{}; return; }
        ProfScope ps(this, PC_LAYERNORM); launch_layernorm(x, rows, g_, b_, a_.p, at, pending_, st_); count_launch(); pending_ = PartialSum{};
    };
    // Q8_0 at large batches: dequantisation runs one layer ahead on its own stream (fork / join through events; inside a graph
    // capture these become plain dependency edges). Layer 0 is dequantised under the front end.
    const bool shadow = shadow_mode(rows);
    if (shadow) {
        NSB_CUDA(cudaEventRecord(ev_lstart_[n_layers], st_));                     // everything of the previous step that read the shadows is behind us
        NSB_CUDA(cudaStreamWaitEvent(st_deq_, ev_lstart_[n_layers], 0));
        pdl_skip_next(); dequant_layer_async(0, st_deq_);
        NSB_CUDA(cudaEventRecord(ev_deq_[0], st_deq_));
    }
    ln(layers_[0].ln[0].as<float>(), layers_[0].ln[1].as<float>());
    // "sub" tap: taken AFTER the first LayerNorm, which folds the split-K planes of the stem projection back into x -- so the
    // tapped run executes exactly the arithmetic of the untapped one (taps only add copies)
    if (debug_) NSB_CUDA(cudaMemcpyAsync(dbg_sub_.p, x, (size_t)rows * D_MODEL * 4, cudaMemcpyDeviceToDevice, st_));
    for (int l = 0; l < n_layers; ++l) {
        LayerW& L = layers_[l];
        if (shadow) {
            NSB_CUDA(cudaEventRecord(ev_lstart_[l], st_));                        // layer l - 1 (the other shadow's reader) is complete at this point
            if (l + 1 < n_layers) {
                NSB_CUDA(cudaStreamWaitEvent(st_deq_, ev_lstart_[l], 0));
                pdl_skip_next(); dequant_layer_async(l + 1, st_deq_);
                NSB_CUDA(cudaEventRecord(ev_deq_[l + 1], st_deq_));
            }
            NSB_CUDA(cudaStreamWaitEvent(st_, ev_deq_[l], 0));                    // this layer's fp16 weights are in place
            cur_shadow_ = shadow_[l & 1].as<char>();
            pdl_skip_next();                                                      // the layer's first GEMM: full dependency (it sits behind a cross-stream wait)
        }
        // FFN1: x += 0.5 * W2 silu(W1 LN(x))                                        (nemo-stream.cpp:603-606)
        if (!(skip & SK_FF)) {
        gemm(a_.p, D_MODEL, L.ff1a, rows, nullptr, big_.p, D_FF, EPI_SILU, 1.f, at);
        gemm_residual(big_.p, D_FF, L.ff1b, rows, x, 0.5f); }
        // MHSA over the ring cache                                                  (:609-615)
        ln(L.ln[2].as<float>(), L.ln[3].as<float>());
        // Small batches (one 128-row tile): with full-K tiles every CTA pulls the whole activation tile (256 KB) and the launch is
        // bound by per-SM L2->SM ingest. Split-K with 64-wide tiles cuts that to 128 + 64 KB (QKV, 2 slices) / 64 + 32 KB
        // (pointwise-1, 4 slices); the fp32 partial planes are summed, in slice order, by the consumer kernel as it loads them.
        const int qkv_planes = split_consumers(rows) ? 2 : 1;
        const int pw1_planes = 1;          // measured (r01_notes.md): 4 slices save 0.75 us in the GEMM and cost 1.2 us in the conv module -> off
        if (!(skip & SK_QKV)) {
            if (qkv_planes == 1) gemm(a_.p, D_MODEL, L.qkv, rows, nullptr, qkv_.p, 3 * D_MODEL, EPI_NONE, 1.f, OUT_F32);
            else gemm_planes(a_.p, D_MODEL, L.qkv, rows, qkv_.p, qkv_planes);
        }
        if (!(skip & SK_ATTN)) {
            AttnArgs aa; aa.qkv = qkv_.as<float>(); aa.planes = qkv_planes; aa.plane_stride = (long long)rows * 3 * D_MODEL;
            const size_t es = kv_elem_size(kv_dtype);
            aa.k_ring = (char*)kv_.p + (size_t)l * 2 * (ATT_L + T) * D_MODEL * es;
            aa.v_ring = (char*)aa.k_ring + (size_t)(ATT_L + T) * D_MODEL * es;
            aa.slot_stride = kv_slot_stride; aa.kv_dtype = kv_dtype; aa.pos_proj = L.pos_proj.p;
            aa.bias_u = L.bias_u.as<float>(); aa.bias_v = L.bias_v.as<float>(); aa.ctx = a_.p; aa.out_type = at;
            aa.slot_of_b = slot; aa.ring_pos = ring_pos_.as<int>(); aa.valid_len = valid_len_.as<int>(); aa.B = B; aa.T = T;
            ProfScope ps(this, PC_ATTENTION); launch_attention(aa, st_); count_launch();
        }
        if (!(skip & SK_OUT)) gemm_residual(a_.p, D_MODEL, L.out, rows, x, 1.f);
        // conv module                                                               (:618-651)
        ln(L.ln[4].as<float>(), L.ln[5].as<float>());
        if (!(skip & SK_PW)) {
            if (pw1_planes == 1) gemm(a_.p, D_MODEL, L.pw1, rows, nullptr, pw1_.p, 2 * D_MODEL, EPI_NONE, 1.f, OUT_F32);
            else gemm_planes(a_.p, D_MODEL, L.pw1, rows, pw1_.p, pw1_planes);
        }
        if (!(skip & SK_CONV)) {
            ConvModArgs ca; ca.pw1 = pw1_.as<float>(); ca.planes = pw1_planes; ca.plane_stride = (long long)rows * 2 * D_MODEL; ca.conv_cache = conv_cache_.as<float>() + (size_t)l * (CONV_K - 1) * D_MODEL;
            ca.slot_stride = cc_slot_stride; ca.par_stride = cc_par_stride; ca.cc_par = cc_par_.as<int>();
            ca.dw_w = L.dw_w.as<float>(); ca.ln_g = L.cln_g.as<float>(); ca.ln_b = L.cln_b.as<float>();
            ca.out = a_.p; ca.out_type = at; ca.slot_of_b = slot; ca.B = B; ca.T = T;
            ProfScope ps(this, PC_CONVMOD); launch_conv_module(ca, st_); count_launch();
        }
        if (!(skip & SK_PW)) gemm_residual(a_.p, D_MODEL, L.pw2, rows, x, 1.f);
        // FFN2                                                                      (:654-657)
        ln(L.ln[6].as<float>(), L.ln[7].as<float>());
        if (!(skip & SK_FF)) {
        gemm(a_.p, D_MODEL, L.ff2a, rows, nullptr, big_.p, D_FF, EPI_SILU, 1.f, at);
        gemm_residual(big_.p, D_FF, L.ff2b, rows, x, 0.5f); }
        // norm_out (:659) fused with the next layer's norm_feed_forward1
        const bool last = l + 1 == n_layers;
        if (skip & SK_LN) pending_ = PartialSum{};
        else { ProfScope ps(this, PC_LAYERNORM);
          launch_layernorm2(x, rows, L.ln[8].as<float>(), L.ln[9].as<float>(), last ? nullptr : layers_[l + 1].ln[0].as<float>(),
                            last ? nullptr : layers_[l + 1].ln[1].as<float>(), last ? nullptr : a_.p, at, pending_, st_);
          count_launch(); pending_ = PartialSum{}; }
        if (debug_) NSB_CUDA(cudaMemcpyAsync(dbg_layers_.as<float>() + (size_t)l * dbg_B_ * T * D_MODEL, x, (size_t)rows * D_MODEL * 4,
                                             cudaMemcpyDeviceToDevice, st_));
    }
    cur_shadow_ = nullptr;
    { ProfScope ps(this, PC_MISC); launch_advance_streams(slot, B, T, ring_pos_.as<int>(), valid_len_.as<int>(), cc_par_.as<int>(), st_); count_launch(); }

    // G: joint.enc for all frames (the decode kernel reads them from this side's buffer)
    if (skip & SK_DECODE) return;
    ProfScope ps_dec(this, PC_DECODE);
    GemmArgs g; g.A = x; g.lda = D_MODEL; g.W = joint_enc_w_.data.p; g.M = rows; g.N = JOINT; g.K = D_MODEL; g.bias = joint_enc_b_.as<float>();
    g.C = side_[side].encp.p; g.ldc = JOINT; g.epi = EPI_NONE;
    // small batches, 3xTF32 (K' = 3072): 20 column tiles cannot keep the machine busy -- six K slices, slice 0 (+ bias) straight into the
    // destination, the other five summed onto it by a small kernel (measured: 25.7 -> ~8 us at 128 rows)
    constexpr int JS = 6;
    const bool jsplit = !strict() && joint_enc_w_.scales.p && rows <= 256 && (size_t)(JS - 1) * rows * JOINT * 4 <= part_.bytes;
    if (jsplit) { g.splits = JS; g.epi = EPI_PARTIAL; g.C0 = side_[side].encp.p; g.C = part_.p; }
    gemm_f32w(g, joint_enc_w_, false);
    if (jsplit) {
        const size_t n4 = (size_t)rows * JOINT / 4;
        launch_k(add_planes_kernel, dim3((unsigned)((n4 + 255) / 256)), dim3(256), 0, st_, side_[side].encp.as<float>(), part_.as<const float>(), JS - 1,
                 (size_t)rows * JOINT, n4);
        count_launch();
    }
}

// Y: the persistent greedy-decode kernel on stream `s`; narrow = a handful of CTA pairs instead of one CTA per SM (decode overlap)
void Engine::run_decode_kernels(int B, int side, cudaStream_t s, bool narrow) {
    ProfScope ps_dec(this, PC_DECODE);
    Side& sd = side_[side];
    DecodeArgs d{};
    d.w.embed = embed_.as<float>();
    for (int l = 0; l < 2; ++l) { d.w.w_ih[l] = lstm_w_[2 * l].as<float>(); d.w.w_hh[l] = lstm_w_[2 * l + 1].as<float>();
                                  d.w.b_ih[l] = lstm_b_[2 * l].as<float>(); d.w.b_hh[l] = lstm_b_[2 * l + 1].as<float>(); }
    d.w.pred_w = pred_w_.as<float>(); d.w.pred_b = pred_b_.as<float>(); d.w.out_w = jout_w_.as<float>(); d.w.out_b = jout_b_.as<float>();
    d.s.hbuf = dec_h_.as<float>(); d.s.cbuf = dec_c_.as<float>(); d.s.par = dec_par_.as<int>();
    d.s.dec_proj = dec_proj_.as<float>(); d.s.prev_token = prev_token_.as<int>(); d.s.cand_valid = cand_valid_.as<int>();
    d.enc_proj = sd.encp.as<float>(); d.slot_of_b = sd.slot.as<int>(); d.B = B; d.T = T;
    d.out_tokens = sd.out_tok.as<int>(); d.out_count = sd.out_cnt.as<int>();
    d.logits_tap = debug_ ? dbg_logits_.as<float>() : nullptr; d.logits_tap_cap = debug_ ? MAX_SYMBOLS * T + T : 0;
    d.logits_tap_n = debug_ ? dbg_logits_n_.as<int>() : nullptr;
    launch_decode(d, sd.sync.p, s, narrow ? decode_narrow_ctas() : 0); count_launch();
}

// ------------------------------------------------------------------------------------------
// bench hooks
// ------------------------------------------------------------------------------------------
void Engine::bench_prepare(int n_streams, const int16_t* pcm, int samples_per_stream, int warm_chunks) {
    if (n_streams < 1 || n_streams > max_streams) throw std::invalid_argument("bench: n_streams out of range");
    const long long need_warm = warm_chunks > 0 ? (long long)HOP * (8LL * T * warm_chunks - 1) + N_FFT / 2 : 0;
    const long long need_all = (long long)HOP * (8LL * T * (warm_chunks + 1) - 1) + N_FFT / 2;
    if (samples_per_stream < need_all) throw std::invalid_argument("bench: need at least " + std::to_string(need_all) + " samples per stream");
    for (int s = 0; s < max_streams; ++s) if (hs_[s].open) hs_[s].open = false;
    std::vector<int> ids;
    for (int i = 0; i < n_streams; ++i) ids.push_back(open_stream());
    for (int i = 0; i < n_streams; ++i) if (need_warm) push_pcm(ids[i], pcm + (size_t)i * samples_per_stream, (int)need_warm);
    while (step() > 0) {}
    // every further full chunk the caller supplied (at most 16) is staged in HBM; the bench steps cycle through them, so the
    // timed steps see different audio (the decode work of a step depends on what the chunk emits)
    int n_chunks = 1;
    while (n_chunks < 16 && samples_per_stream >= (long long)HOP * (8LL * T * (warm_chunks + n_chunks + 1) - 1) + N_FFT / 2) ++n_chunks;
    const long long need_stage = (long long)HOP * (8LL * T * (warm_chunks + n_chunks) - 1) + N_FFT / 2;
    for (int i = 0; i < n_streams; ++i) push_pcm(ids[i], pcm + (size_t)i * samples_per_stream + need_warm, (int)(need_stage - need_warm));
    bench_pcm_.alloc((size_t)n_chunks * n_streams * rl_ * 2, false);
    int16_t* hp = io_[0].h_pcm.as<int16_t>(); int* hsl = io_[0].h_slot.as<int>();
    for (int k = 0; k < n_chunks; ++k) {
        for (int b = 0; b < n_streams; ++b) {
            HostStream& h = hs_[ids[b]];
            if (k == 0 && !ready(ids[b])) throw std::runtime_error("bench: stream not ready after staging");
            h.chunk_idx += k;                                                     // row of chunk (current + k); host state is restored right away
            hs_stage_row(h, T, rl_, hp + (size_t)b * rl_);
            h.chunk_idx -= k;
            hsl[b] = ids[b];
        }
        h2d_sync((char*)bench_pcm_.p + (size_t)k * n_streams * rl_ * 2, hp, (size_t)n_streams * rl_ * 2);
    }
    for (Side& sd : side_) h2d_sync(sd.slot.p, hsl, (size_t)n_streams * 4);
    bench_B_ = n_streams; bench_n_ = n_chunks; bench_i_ = 0;
}

const int16_t* Engine::bench_next_pcm() {
    const int16_t* p = bench_pcm_.as<int16_t>() + (size_t)(bench_i_ % bench_n_) * bench_B_ * rl_;
    bench_i_ += 1;
    return p;
}

float Engine::bench_step() {
    if (!bench_B_) throw std::runtime_error("bench_step before bench_prepare");
    collect_all();
    NSB_CUDA(cudaSetDevice(device_));
    NSB_CUDA(cudaEventRecord(ev0_, st_));
    cudaStream_t tail = run_step(bench_B_, bench_next_pcm(), side_acquire(), false);
    NSB_CUDA(cudaEventRecord(ev1_, tail));
    NSB_CUDA(cudaEventSynchronize(ev1_));
    float ms = 0.f; NSB_CUDA(cudaEventElapsedTime(&ms, ev0_, ev1_));
    stats.steps += 1; stats.chunks += bench_B_; stats.device_ms += ms; stats.last_step_ms = ms;
    return ms;
}

float Engine::bench_steps(int n, float* ms_each) {
    if (!bench_B_) throw std::runtime_error("bench_steps before bench_prepare");
    if (n < 1) throw std::invalid_argument("bench_steps: n < 1");
    collect_all();
    NSB_CUDA(cudaSetDevice(device_));
    ev_used_ = 0;
    std::vector<cudaEvent_t> ev((size_t)n + 1);
    for (int i = 0; i <= n; ++i) ev[i] = prof_event();
    NSB_CUDA(cudaEventRecord(ev[0], st_));
    // with decode overlap the event after step i sits behind its DECODE (other stream): the encoder of step i + 1 is already running
    for (int i = 0; i < n; ++i) { cudaStream_t tail = run_step(bench_B_, bench_next_pcm(), side_acquire(), n > 1); NSB_CUDA(cudaEventRecord(ev[i + 1], tail)); }
    NSB_CUDA(cudaEventSynchronize(ev[n]));
    float total = 0.f; NSB_CUDA(cudaEventElapsedTime(&total, ev[0], ev[n]));
    for (int i = 0; i < n; ++i) {
        float ms = 0.f; NSB_CUDA(cudaEventElapsedTime(&ms, ev[i], ev[i + 1]));
        if (ms_each) ms_each[i] = ms;
    }
    stats.steps += n; stats.chunks += (long long)n * bench_B_; stats.device_ms += total; stats.last_step_ms = total / n;
    ev_used_ = 0;
    return total;
}

float Engine::bench_gemm(int kind, int rows, int bn, int stages, int splits, int rotate, int iters) {
    if (strict()) throw std::runtime_error("bench_gemm: tensor-core modes only");
    if (rows < 1 || rows > max_streams * T || kind < 0 || kind > 5) throw std::invalid_argument("bench_gemm: bad arguments");
    NSB_CUDA(cudaSetDevice(device_));
    const bool use_shadow = splits < 0 && shadow_mode(rows) && n_layers >= 2;
    auto pick = [&](LayerW& L) -> Weight& { switch (kind) { case 0: return L.ff1a; case 1: return L.ff1b; case 2: return L.qkv; case 3: return L.out; case 4: return L.pw1; default: return L.pw2; } };
    auto run = [&]() {
        for (int l = 0; l < n_layers; ++l) {
            Weight& W = pick(layers_[l]);
            if (splits < 0) {
                // the step's own launch for this matrix: same tile choice, split-K rule and epilogue; Q8_0 at large batches: on the fp16
                // shadow a layer-ahead dequantisation leaves (two shadows, filled once below: these launches time the GEMM alone)
                if (use_shadow) cur_shadow_ = shadow_[l & 1].as<char>();
                switch (kind) {
                    case 0: gemm(a_.p, D_MODEL, W, rows, nullptr, big_.p, D_FF, EPI_SILU, 1.f, act_type()); break;
                    case 2: if (split_consumers(rows)) gemm_planes(a_.p, D_MODEL, W, rows, qkv_.p, 2);
                            else gemm(a_.p, D_MODEL, W, rows, nullptr, qkv_.p, 3 * D_MODEL, EPI_NONE, 1.f, OUT_F32);
                            break;
                    case 4: gemm(a_.p, D_MODEL, W, rows, nullptr, pw1_.p, 2 * D_MODEL, EPI_NONE, 1.f, OUT_F32); break;
                    case 1: gemm_residual(big_.p, D_FF, W, rows, x_.as<float>(), 0.5f); break;
                    default: gemm_residual(a_.p, D_MODEL, W, rows, x_.as<float>(), 1.f); break;
                }
                pending_ = PartialSum{}; cur_shadow_ = nullptr;
                continue;
            }
            GemmArgs a; a.A = W.n_in == D_FF ? big_.p : a_.p; a.lda = W.n_in; a.W = W.data.p; a.w_scales = W.scales.p; a.q4 = W.q4; a.M = rows; a.N = W.n_out; a.K = W.n_in;
            a.force_bn = bn; a.force_stages = stages; a.rotate = rotate; a.splits = splits; a.ldc = W.n_out; a.pair = splits == 1;
            if (splits > 1) { a.C = part_.p; a.epi = EPI_PARTIAL; a.out_type = OUT_F32; }
            else if (W.n_out == D_FF) { a.C = big_.p; a.epi = EPI_SILU; a.out_type = act_type(); }
            else { a.C = qkv_.p; a.epi = EPI_NONE; a.out_type = OUT_F32; }
            q8_predequant(W, rows, a);                    // Q8_0 mode, >= 512 rows: the dequantisation pass is part of the launch, as in the step
            launch_gemm_tc(a, act_type(), st_);
        }
    };
    if (splits > 1 && (size_t)splits * rows * pick(layers_[0]).n_out * 4 > part_.bytes) throw std::invalid_argument("bench_gemm: split workspace too small");
    if (use_shadow) { collect_all(); join_decode_stream(); dequant_layer_async(0, st_); dequant_layer_async(1, st_); NSB_CUDA(cudaStreamSynchronize(st_)); }
    run();
    // One pass over the layers is captured into a CUDA graph, as the step is: stream launches of ~3 us kernels (two tensor-map
    // encodes + cudaLaunchKernelEx each) would time the host, not the kernel. NSB_BENCH_GEMM_GRAPH=0: plain stream launches.
    static const bool use_graph = [] { const char* e = getenv("NSB_BENCH_GEMM_GRAPH"); return !(e && e[0] == '0'); }();
    cudaGraphExec_t exec = nullptr;
    if (use_graph) {
        cudaGraph_t graph = nullptr;
        NSB_CUDA(cudaStreamBeginCapture(st_, cudaStreamCaptureModeRelaxed));
        try { run(); } catch (...) { cudaStreamEndCapture(st_, &graph); if (graph) cudaGraphDestroy(graph); throw; }
        NSB_CUDA(cudaStreamEndCapture(st_, &graph));
        const cudaError_t err = cudaGraphInstantiate(&exec, graph, 0);
        cudaGraphDestroy(graph);
        if (err != cudaSuccess) throw CudaError(std::string("bench_gemm: cudaGraphInstantiate: ") + cudaGetErrorString(err));
        NSB_CUDA(cudaGraphLaunch(exec, st_));
    }
    NSB_CUDA(cudaEventRecord(ev0_, st_));
    for (int i = 0; i < iters; ++i) { if (exec) { NSB_CUDA(cudaGraphLaunch(exec, st_)); } else { run(); } }
    NSB_CUDA(cudaEventRecord(ev1_, st_));
    NSB_CUDA(cudaEventSynchronize(ev1_));
    float ms = 0.f; NSB_CUDA(cudaEventElapsedTime(&ms, ev0_, ev1_));
    if (exec) cudaGraphExecDestroy(exec);
    return 1e3f * ms / (float)(iters * n_layers);
}

void Engine::trace_enable(int cap) {
    NSB_CUDA(cudaSetDevice(device_));
    NSB_CUDA(cudaStreamSynchronize(st_));
    TraceBuf* p = nullptr;
    if (cap > 0) {
        trace_.alloc(sizeof(TraceBuf) + (size_t)cap * sizeof(TraceRec));
        const unsigned hdr[4] = {0u, (unsigned)cap, 0u, 0u};
        h2d_sync(trace_.p, hdr, sizeof(hdr));
        p = trace_.as<TraceBuf>();
    }
    trace_cap_ = cap > 0 ? cap : 0;
    trace_bind_frontend(p); trace_bind_layer(p); trace_bind_simt(p); trace_bind_gemm_tc(p); trace_bind_decode(p);
    NSB_CUDA(cudaDeviceSynchronize());
}

int Engine::trace_fetch(TraceRec* out, int cap) {
    if (!trace_cap_) return 0;
    NSB_CUDA(cudaSetDevice(device_));
    NSB_CUDA(cudaStreamSynchronize(st_));
    unsigned n = 0;
    NSB_CUDA(cudaMemcpy(&n, trace_.p, 4, cudaMemcpyDeviceToHost));
    const int m = (int)std::min<unsigned>(std::min<unsigned>(n, (unsigned)trace_cap_), (unsigned)std::max(cap, 0));
    if (m > 0) NSB_CUDA(cudaMemcpy(out, (char*)trace_.p + offsetof(TraceBuf, rec), (size_t)m * sizeof(TraceRec), cudaMemcpyDeviceToHost));
    const unsigned zero = 0; h2d_sync(trace_.p, &zero, 4);
    return m;
}

cudaEvent_t Engine::prof_event() {
    if (ev_used_ == ev_pool_.size()) { cudaEvent_t e; NSB_CUDA(cudaEventCreate(&e)); ev_pool_.push_back(e); }
    return ev_pool_[ev_used_++];
}

float Engine::bench_profile(float* ms_per_class, int* launches_per_class) {
    if (!bench_B_) throw std::runtime_error("bench_profile before bench_prepare");
    NSB_CUDA(cudaSetDevice(device_));
    join_decode_stream();
    prof_.clear(); ev_used_ = 0; profiling_ = true;
    NSB_CUDA(cudaEventRecord(ev0_, st_));
    { const int side = side_acquire(); run_encoder_kernels(bench_B_, bench_pcm_.as<int16_t>(), side); run_decode_kernels(bench_B_, side, st_, false); side_next_ = (side + 1) % MAX_INFLIGHT; }
    NSB_CUDA(cudaEventRecord(ev1_, st_));
    profiling_ = false;
    NSB_CUDA(cudaEventSynchronize(ev1_));
    for (int c = 0; c < PC_COUNT; ++c) { ms_per_class[c] = 0.f; launches_per_class[c] = 0; }
    for (const ProfRec& r : prof_) { float ms = 0.f; NSB_CUDA(cudaEventElapsedTime(&ms, r.a, r.b)); ms_per_class[r.cls] += ms; launches_per_class[r.cls] += 1; }
    float total = 0.f; NSB_CUDA(cudaEventElapsedTime(&total, ev0_, ev1_));
    return total;
}

// ------------------------------------------------------------------------------------------
// debug taps + stand-alone operators
// ------------------------------------------------------------------------------------------
void Engine::debug_enable(bool on) {
    NSB_CUDA(cudaSetDevice(device_));
    collect_all(); join_decode_stream();
    debug_ = on;
    if (!on) return;
    dbg_B_ = max_streams;
    const size_t rows = (size_t)dbg_B_ * T;
    dbg_mel_.alloc((size_t)dbg_B_ * (PRE_CACHE + 8 * T) * N_MELS * 4);
    dbg_sub_.alloc(rows * D_MODEL * 4);
    dbg_layers_.alloc((size_t)n_layers * rows * D_MODEL * 4);
    dbg_logits_.alloc((size_t)(MAX_SYMBOLS * T + T) * VOCAB * 4);
    dbg_logits_n_.alloc(4);
}

long long Engine::debug_get(const std::string& name, float* out, size_t cap) {
    if (name == "x") {
        // Encoder output of the most recently LAUNCHED step, read straight out of the step workspace: needs no tap mode, so it
        // observes the production path (CUDA graph replay, PDL, split-K folded into LayerNorm) unchanged. Rows = that step's batch
        // order. The caller must read it before launching the next step.
        NSB_CUDA(cudaSetDevice(device_));
        NSB_CUDA(cudaStreamSynchronize(st_));
        const size_t n = std::min((size_t)last_B_ * T * D_MODEL, cap);
        if (n) NSB_CUDA(cudaMemcpy(out, x_.p, n * 4, cudaMemcpyDeviceToHost));
        return (long long)n;
    }
    if (!debug_) throw std::runtime_error("debug taps are not enabled");
    NSB_CUDA(cudaSetDevice(device_));
    NSB_CUDA(cudaStreamSynchronize(st_));
    const void* src = nullptr; size_t n = 0;
    const size_t rows_all = (size_t)dbg_B_ * T;
    if (name == "mel") { src = dbg_mel_.p; n = (size_t)dbg_B_ * (PRE_CACHE + 8 * T) * N_MELS; }
    else if (name == "sub") { src = dbg_sub_.p; n = rows_all * D_MODEL; }
    else if (name == "enc") { src = dbg_layers_.as<float>() + (size_t)(n_layers - 1) * rows_all * D_MODEL; n = rows_all * D_MODEL; }
    else if (name.rfind("layer.", 0) == 0) {
        const int l = atoi(name.c_str() + 6);
        if (l < 0 || l >= n_layers) throw std::invalid_argument("layer index");
        src = dbg_layers_.as<float>() + (size_t)l * rows_all * D_MODEL; n = rows_all * D_MODEL;
    } else if (name == "logits") {
        int ne = 0; NSB_CUDA(cudaMemcpy(&ne, dbg_logits_n_.p, 4, cudaMemcpyDeviceToHost));
        ne = std::min(ne, MAX_SYMBOLS * T + T);
        src = dbg_logits_.p; n = (size_t)ne * VOCAB;
    } else throw std::invalid_argument("unknown tap '" + name + "'");
    n = std::min(n, cap);
    NSB_CUDA(cudaMemcpy(out, src, n * 4, cudaMemcpyDeviceToHost));
    return (long long)n;
}

long long Engine::debug_get_cache(int stream, int which, int layer, float* out, size_t cap) {
    if (stream < 0 || stream >= max_streams || layer < 0 || layer >= n_layers) throw std::invalid_argument("bad stream/layer");
    NSB_CUDA(cudaSetDevice(device_));
    NSB_CUDA(cudaStreamSynchronize(st_));
    if (which == 2) {
        const size_t n = (size_t)(CONV_K - 1) * D_MODEL; if (cap < n) return -(long long)n;
        int par = 0; NSB_CUDA(cudaMemcpy(&par, cc_par_.as<int>() + stream, 4, cudaMemcpyDeviceToHost));      // the parity the last step wrote = the current one
        NSB_CUDA(cudaMemcpy(out, conv_cache_.as<float>() + (((size_t)stream * 2 + (par & 1)) * n_layers + layer) * n, n * 4, cudaMemcpyDeviceToHost));
        return (long long)n;
    }
    // K / V: return the 70 cache rows in logical order (oldest first), as the reference's rolled cache holds them
    const int Cap = ATT_L + T; const size_t es = kv_elem_size(kv_dtype);
    const size_t n = (size_t)ATT_L * D_MODEL; if (cap < n) return -(long long)n;
    std::vector<uint8_t> raw((size_t)Cap * D_MODEL * es);
    const size_t off = (((size_t)stream * n_layers + layer) * 2 + (which ? 1 : 0)) * Cap * D_MODEL * es;
    NSB_CUDA(cudaMemcpy(raw.data(), (char*)kv_.p + off, raw.size(), cudaMemcpyDeviceToHost));
    int w = 0; NSB_CUDA(cudaMemcpy(&w, ring_pos_.as<int>() + stream, 4, cudaMemcpyDeviceToHost));
    for (int j = 0; j < ATT_L; ++j) {
        const int r = (w + Cap - ATT_L + j) % Cap;           // after advance: the 70 rows before the write position
        for (int c = 0; c < D_MODEL; ++c) {
            const size_t i = (size_t)r * D_MODEL + c; float v;
            if (kv_dtype == 0) v = ((const float*)raw.data())[i];
            else if (kv_dtype == 1) v = half_bits_to_float(((const uint16_t*)raw.data())[i]);
            else { uint32_t u = (uint32_t)((const uint16_t*)raw.data())[i] << 16; memcpy(&v, &u, 4); }
            out[(size_t)j * D_MODEL + c] = v;
        }
    }
    return (long long)n;
}

long long Engine::op_logmel(const int16_t* pcm, int n_streams, int n_samples, float* out, size_t cap) {
    if (n_streams < 1 || n_samples < 1) throw std::invalid_argument("op_logmel: empty input");
    NSB_CUDA(cudaSetDevice(device_));
    const long long avail = N_FFT / 2 + (long long)n_samples;
    const int n_frames = avail < N_FFT ? 0 : (int)((avail - N_FFT + HOP) / HOP);     // preprocessor.cpp:320-328
    if (n_frames == 0) return 0;
    if (cap < (size_t)n_streams * n_frames * N_MELS) return -(long long)((size_t)n_streams * n_frames * N_MELS);
    const int row = 1 + N_FFT / 2 + n_samples;
    std::vector<int16_t> h((size_t)n_streams * row, 0);
    for (int s = 0; s < n_streams; ++s) memcpy(&h[(size_t)s * row + 1 + N_FFT / 2], pcm + (size_t)s * n_samples, (size_t)n_samples * 2);
    DevBuf d_in, d_out; d_in.alloc(h.size() * 2, false); d_out.alloc((size_t)n_streams * n_frames * N_MELS * 4, false);
    h2d_sync(d_in.p, h.data(), h.size() * 2);
    launch_logmel(d_in.as<int16_t>(), row, n_streams, n_frames, window_.as<float>(), cos_t_.as<float>(), sin_t_.as<float>(), fb_t_.as<float>(),
                  d_out.as<float>(), (size_t)n_frames * N_MELS, st_);
    count_launch();
    NSB_CUDA(cudaStreamSynchronize(st_));
    NSB_CUDA(cudaMemcpy(out, d_out.p, d_out.bytes, cudaMemcpyDeviceToHost));
    return n_frames;
}

// ------------------------------------------------------------------------------------------
// Non-streaming batch path (SURVEY 8f.1), validated on hardware against the checker (orc_transcribe_full) and the fixture made by the
// reference's own compiled modules (tests/golden/batch_ref_L2.npz; tests/test_zz_batch_path.py: 2 layers and 24 layers x 30 s). Everything
// except the full-context attention kernel and the un-chunked stem variant is the streaming step's own kernels: a non-cached conformer
// layer is the cached one with an empty cache (zeroed conv state = the causal pad of nemo-ggml.cpp:706-707). Private workspace and a
// private state slot: open streams are not disturbed.
// ------------------------------------------------------------------------------------------
void Engine::ensure_full_pos(int frames) {
    if (frames <= full_pos_cap_) return;
    const int cap = std::max(frames, 256), n_rel = 2 * cap - 1;
    ensure_q8s_scratch(n_rel);                  // row r <-> relative position r - (cap - 1) = query - key
    GgufFile g; g.open(gguf_path_);
    std::vector<float> tab((size_t)n_rel * D_MODEL);
    for (int r = 0; r < n_rel; ++r) pos_emb_row(r - (cap - 1), &tab[(size_t)r * D_MODEL]);
    DevBuf d_tab; upload(d_tab, tab);
    DevBuf d_a; const void* A = d_tab.p;
    if (act_type() != OUT_F32) { d_a.alloc(tab.size() * 2, false); convert_to(d_tab.as<float>(), d_a.p, tab.size(), act_type(), st_); A = d_a.p; }
    full_pos_.clear(); full_pos_.resize((size_t)n_layers);
    DevBuf tmp; if (kv_dtype != 0) tmp.alloc((size_t)n_rel * D_MODEL * 4, false);
    for (int l = 0; l < n_layers; ++l) {
        const std::string n = "encoder.layers." + std::to_string(l) + ".self_attn.linear_pos.weight";
        Weight wpos; load_layer_matrix(wpos, g, n, {n}, D_MODEL, D_MODEL);
        full_pos_[l].alloc((size_t)n_rel * D_MODEL * kv_elem_size(kv_dtype), false);
        gemm(A, D_MODEL, wpos, n_rel, nullptr, kv_dtype == 0 ? full_pos_[l].p : tmp.p, D_MODEL, EPI_NONE, 1.f, OUT_F32);
        if (kv_dtype != 0) convert_to(tmp.as<float>(), full_pos_[l].p, (size_t)n_rel * D_MODEL, kv_dtype == 1 ? OUT_F16 : OUT_BF16, st_);
        NSB_CUDA(cudaStreamSynchronize(st_));                                     // wpos dies at the end of the iteration
    }
    full_pos_cap_ = cap;
}

void Engine::ensure_batch_work(int rows, int t2) {
    const size_t sp = (!strict() && tf32x3_enabled()) ? 2 : 1;
    const size_t pix = (size_t)t2 * 33 * SUB_CH * 4;
    if (rows <= bw_.rows && bw_.pw.bytes >= pix) return;
    NSB_CUDA(cudaStreamSynchronize(st_));
    const size_t r = (size_t)std::max(rows, 64);
    bw_.dw.alloc(sp * pix, false); bw_.pw.alloc(pix, false);
    if (sp == 2) bw_.a3.alloc(r * SUB_W * SUB_CH * 2 * 4, false);
    bw_.x.alloc(r * D_MODEL * 4, false); bw_.a.alloc(r * D_MODEL * act_size(), false); bw_.big.alloc(r * D_FF * act_size(), false);
    bw_.qkv.alloc(r * 3 * D_MODEL * 4, false); bw_.pw1.alloc(r * 2 * D_MODEL * 4, false); bw_.encp.alloc(r * JOINT * 4, false);
    bw_.part.alloc(std::max((size_t)MAX_SPLITS * std::min<size_t>(r, 1024), 4 * r) * D_MODEL * 4, false);
    bw_.out_tok.alloc(r * MAX_SYMBOLS * 4, false); bw_.out_frm.alloc(r * MAX_SYMBOLS * 4, false);
    bw_.rows = (int)r;
    ensure_q8s_scratch((int)r);
}
void Engine::swap_batch_work() {
    std::swap(dw_, bw_.dw); std::swap(pw_, bw_.pw); std::swap(a3_, bw_.a3); std::swap(x_, bw_.x); std::swap(a_, bw_.a); std::swap(big_, bw_.big);
    std::swap(qkv_, bw_.qkv); std::swap(pw1_, bw_.pw1); std::swap(encp_, bw_.encp); std::swap(part_, bw_.part); std::swap(out_tok_, bw_.out_tok);
}

long long Engine::transcribe_full(const int16_t* pcm, int n_samples, int32_t* tokens, int32_t* token_frames, int cap, int* n_frames, float* enc_out, size_t enc_cap) {
    if (!pcm || n_samples < 1 || (!tokens && cap > 0) || cap < 0) throw std::invalid_argument("transcribe_full: bad arguments");
    collect_all();
    NSB_CUDA(cudaSetDevice(device_));
    if (n_frames) *n_frames = 0;
    const long long avail = N_FFT / 2 + (long long)n_samples;
    const int M = avail < N_FFT ? 0 : (int)((avail - N_FFT + HOP) / HOP);         // preprocessor.cpp:320-328
    if (M == 0) return 0;
    const int t1 = M / 2 + 1, t2 = t1 / 2 + 1, t3 = t2 / 2 + 1, Tq = t3;          // three 3x3 s2 convs with (2, 1) padding (nemo-ggml.cpp:828-836)
    if (Tq > 2048) throw std::invalid_argument("transcribe_full: more than 2048 encoder frames (the reference's positional table, nemo-ggml.cpp:196)");
    if (enc_out && enc_cap < (size_t)Tq * D_MODEL) return -(long long)((size_t)Tq * D_MODEL);
    join_decode_stream();
    ensure_full_pos(Tq);
    ensure_batch_work(Tq, t2);
    const int slot = max_streams;                                                 // the batch path's private slot
    zero_slot(slot);                                                              // zeroed conv state, decoder state, prev_token = blank
    swap_batch_work();                                                            // the step workspace (and the graphs captured on it) stays untouched
    struct Release { Engine* e; ~Release() { e->swap_batch_work(); } } release{this};

    // P: log-mel of the whole utterance (row = x[-1] = 0, the 256-zero left pad, the samples: preprocessor.cpp:220-221,349-356)
    const int row = 1 + N_FFT / 2 + n_samples;
    std::vector<int16_t> h((size_t)row, 0);
    memcpy(&h[1 + N_FFT / 2], pcm, (size_t)n_samples * 2);
    DevBuf d_in, d_mel; d_in.alloc(h.size() * 2, false); d_mel.alloc((size_t)M * N_MELS * 4, false);
    h2d_sync(d_in.p, h.data(), h.size() * 2);
    h2d_sync(d_slot_.p, &slot, 4);
    launch_logmel(d_in.as<int16_t>(), row, 1, M, window_.as<float>(), cos_t_.as<float>(), sin_t_.as<float>(), fb_t_.as<float>(), d_mel.as<float>(),
                  (size_t)M * N_MELS, st_);
    count_launch();

    // S: subsampling of the whole image, no carried frames, nothing dropped (build_conv_subsampling, nemo-ggml.cpp:877-952)
    const int at = act_type(), rows = Tq;
    const int* slot_dev = d_slot_.as<int>();
    float* x = x_.as<float>();
    pending_ = PartialSum{};
    const bool tc = !strict();
    const int split = tc && c3_w_.scales.p ? 1 : 0;
    launch_stem_conv0_dw_full(d_mel.as<float>(), 1, M, c0_w_.as<float>(), c0_b_.as<float>(), c2_w_.as<float>(), c2_b_.as<float>(), dw_.as<float>(), st_, split);
    count_launch();
    {
        GemmArgs g; g.A = dw_.p; g.lda = SUB_CH; g.W = c3_w_.data.p; g.M = t2 * 33; g.N = SUB_CH; g.K = SUB_CH; g.bias = c3_b_.as<float>();
        g.C = pw_.p; g.ldc = SUB_CH; g.epi = EPI_RELU; gemm_f32w(g, c3_w_, split);
    }
    launch_dwconv_s2(pw_.as<float>(), 1, t2, 33, c5_w_.as<float>(), c5_b_.as<float>(), dw_.as<float>(), st_, split); count_launch();
    {
        GemmArgs g; g.A = dw_.p; g.lda = SUB_CH; g.W = c6_w_.data.p; g.M = t3 * SUB_W; g.N = SUB_CH; g.K = SUB_CH; g.bias = c6_b_.as<float>();
        g.C = pw_.p; g.ldc = SUB_CH; g.epi = EPI_RELU; gemm_f32w(g, c6_w_, split);
    }
    {
        GemmArgs g; g.A = pw_.p; g.lda = SUB_W * SUB_CH; g.W = sub_out_w_.data.p; g.M = rows; g.N = D_MODEL; g.K = SUB_W * SUB_CH; g.bias = out_b_.as<float>();
        g.C = x; g.ldc = D_MODEL; g.epi = EPI_NONE; gemm_f32w(g, sub_out_w_, false);
    }

    // L: the layers of build_conformer_layer (nemo-ggml.cpp:768-818) on the cached-layer kernels
    const long long cc_par_stride = (long long)n_layers * (CONV_K - 1) * D_MODEL, cc_slot_stride = 2 * cc_par_stride;
    auto ln = [&](const float* g_, const float* b_) { launch_layernorm(x, rows, g_, b_, a_.p, at, pending_, st_); count_launch(); pending_ = PartialSum{}; };
    ln(layers_[0].ln[0].as<float>(), layers_[0].ln[1].as<float>());
    for (int l = 0; l < n_layers; ++l) {
        LayerW& L = layers_[l];
        gemm(a_.p, D_MODEL, L.ff1a, rows, nullptr, big_.p, D_FF, EPI_SILU, 1.f, at);
        gemm_residual(big_.p, D_FF, L.ff1b, rows, x, 0.5f);
        ln(L.ln[2].as<float>(), L.ln[3].as<float>());
        gemm(a_.p, D_MODEL, L.qkv, rows, nullptr, qkv_.p, 3 * D_MODEL, EPI_NONE, 1.f, OUT_F32);
        {
            AttnFullArgs fa; fa.qkv = qkv_.as<float>(); fa.pos_proj = full_pos_[l].p; fa.pos_center = full_pos_cap_ - 1; fa.kv_dtype = kv_dtype;
            fa.bias_u = L.bias_u.as<float>(); fa.bias_v = L.bias_v.as<float>(); fa.ctx = a_.p; fa.out_type = at; fa.T = rows;
            launch_attention_full(fa, st_); count_launch();
        }
        gemm_residual(a_.p, D_MODEL, L.out, rows, x, 1.f);
        ln(L.ln[4].as<float>(), L.ln[5].as<float>());
        gemm(a_.p, D_MODEL, L.pw1, rows, nullptr, pw1_.p, 2 * D_MODEL, EPI_NONE, 1.f, OUT_F32);
        {
            ConvModArgs ca; ca.pw1 = pw1_.as<float>(); ca.planes = 1; ca.plane_stride = (long long)rows * 2 * D_MODEL;
            ca.conv_cache = conv_cache_.as<float>() + (size_t)l * (CONV_K - 1) * D_MODEL; ca.slot_stride = cc_slot_stride;
            ca.par_stride = cc_par_stride; ca.cc_par = cc_par_.as<int>();
            ca.dw_w = L.dw_w.as<float>(); ca.ln_g = L.cln_g.as<float>(); ca.ln_b = L.cln_b.as<float>();
            ca.out = a_.p; ca.out_type = at; ca.slot_of_b = slot_dev; ca.B = 1; ca.T = rows;
            launch_conv_module(ca, st_); count_launch();
        }
        gemm_residual(a_.p, D_MODEL, L.pw2, rows, x, 1.f);
        ln(L.ln[6].as<float>(), L.ln[7].as<float>());
        gemm(a_.p, D_MODEL, L.ff2a, rows, nullptr, big_.p, D_FF, EPI_SILU, 1.f, at);
        gemm_residual(big_.p, D_FF, L.ff2b, rows, x, 0.5f);
        const bool last = l + 1 == n_layers;
        launch_layernorm2(x, rows, L.ln[8].as<float>(), L.ln[9].as<float>(), last ? nullptr : layers_[l + 1].ln[0].as<float>(),
                          last ? nullptr : layers_[l + 1].ln[1].as<float>(), last ? nullptr : a_.p, at, pending_, st_);
        count_launch(); pending_ = PartialSum{};
    }

    // G/Y: greedy_decode (nemo-ggml.cpp:1109-1258) from a fresh decoder state over all frames
    {
        GemmArgs g; g.A = x; g.lda = D_MODEL; g.W = joint_enc_w_.data.p; g.M = rows; g.N = JOINT; g.K = D_MODEL; g.bias = joint_enc_b_.as<float>();
        g.C = encp_.p; g.ldc = JOINT; g.epi = EPI_NONE; gemm_f32w(g, joint_enc_w_, false);
    }
    DecodeArgs d{};
    d.w.embed = embed_.as<float>();
    for (int l = 0; l < 2; ++l) { d.w.w_ih[l] = lstm_w_[2 * l].as<float>(); d.w.w_hh[l] = lstm_w_[2 * l + 1].as<float>();
                                  d.w.b_ih[l] = lstm_b_[2 * l].as<float>(); d.w.b_hh[l] = lstm_b_[2 * l + 1].as<float>(); }
    d.w.pred_w = pred_w_.as<float>(); d.w.pred_b = pred_b_.as<float>(); d.w.out_w = jout_w_.as<float>(); d.w.out_b = jout_b_.as<float>();
    d.s.hbuf = dec_h_.as<float>(); d.s.cbuf = dec_c_.as<float>(); d.s.par = dec_par_.as<int>();
    d.s.dec_proj = dec_proj_.as<float>(); d.s.prev_token = prev_token_.as<int>(); d.s.cand_valid = cand_valid_.as<int>();
    d.enc_proj = encp_.as<float>(); d.slot_of_b = slot_dev; d.B = 1; d.T = rows;
    d.out_tokens = out_tok_.as<int>(); d.out_count = out_cnt_.as<int>(); d.out_frames = bw_.out_frm.as<int>();
    launch_decode(d, dec_sync_.p, st_); count_launch();
    NSB_CUDA(cudaStreamSynchronize(st_));

    int n_tok = 0;
    NSB_CUDA(cudaMemcpy(&n_tok, out_cnt_.p, 4, cudaMemcpyDeviceToHost));
    n_tok = std::max(0, std::min(n_tok, MAX_SYMBOLS * rows));
    if (std::min(n_tok, cap) > 0) NSB_CUDA(cudaMemcpy(tokens, out_tok_.p, (size_t)std::min(n_tok, cap) * 4, cudaMemcpyDeviceToHost));
    if (token_frames && std::min(n_tok, cap) > 0) NSB_CUDA(cudaMemcpy(token_frames, bw_.out_frm.p, (size_t)std::min(n_tok, cap) * 4, cudaMemcpyDeviceToHost));
    if (enc_out) NSB_CUDA(cudaMemcpy(enc_out, x, (size_t)rows * D_MODEL * 4, cudaMemcpyDeviceToHost));
    if (n_frames) *n_frames = rows;
    stats.chunks += 1;
    return n_tok;
}

// The op_* GEMMs below take the weight's A operand the way the step's producers leave it: rounded to the activation type for the
// per-layer matrices, plain f32 for the F32 matrices (3xTF32 splits it, strict modes run SIMT fp32).
const Weight& Engine::op_weight(const std::string& name) const {
    auto it = named_.find(name);
    if (it == named_.end()) throw std::invalid_argument("op_gemm: unknown weight '" + name + "'");
    return *it->second;
}
const void* Engine::op_operand(const Weight& W, const float* xh, int rows, DevBuf& dx, DevBuf& da) {
    dx.alloc((size_t)rows * W.n_in * 4, false);
    h2d_sync(dx.p, xh, dx.bytes);
    if (W.f32 || act_type() == OUT_F32) return dx.p;
    da.alloc((size_t)rows * W.n_in * 2, false);
    convert_to(dx.as<float>(), da.p, (size_t)rows * W.n_in, act_type(), st_);
    return da.p;
}
// F32 matrices: gemm_f32w splits A into a3_, which the step sizes for its own batch; a larger operator call borrows a scratch of its
// own for the duration (a3_ itself stays where the captured step graphs expect it)
struct Engine::SplitScratch {
    Engine* e; DevBuf tmp; bool swapped = false;
    SplitScratch(Engine* e_, const Weight& W, int rows) : e(e_) {
        const size_t need = (size_t)rows * 2 * W.n_in * 4;
        if (!W.f32 || !W.scales.p || e->a3_.bytes >= need) return;
        tmp.alloc(need, false); std::swap(e->a3_, tmp); swapped = true;
    }
    ~SplitScratch() { if (swapped) { cudaStreamSynchronize(e->st_); std::swap(e->a3_, tmp); } }
};

long long Engine::op_gemm(const std::string& name, const float* xh, int rows, float* y, size_t cap) {
    const Weight& W = op_weight(name);
    NSB_CUDA(cudaSetDevice(device_));
    if (cap < (size_t)rows * W.n_out) return -(long long)((size_t)rows * W.n_out);
    ensure_q8s_scratch(rows);
    DevBuf dx, da, dy; dy.alloc((size_t)rows * W.n_out * 4, false);
    const void* A = op_operand(W, xh, rows, dx, da);
    if (W.f32) {
        SplitScratch sc(this, W, rows);
        GemmArgs g; g.A = A; g.lda = W.n_in; g.W = W.data.p; g.M = rows; g.N = W.n_out; g.K = W.n_in; g.C = dy.p; g.ldc = W.n_out; g.epi = EPI_NONE;
        gemm_f32w(g, W, false);
    } else gemm(A, W.n_in, W, rows, nullptr, dy.p, W.n_out, EPI_NONE, 1.f, OUT_F32);
    NSB_CUDA(cudaStreamSynchronize(st_));
    NSB_CUDA(cudaMemcpy(y, dy.p, dy.bytes, cudaMemcpyDeviceToHost));
    return W.n_out;
}

namespace {
constexpr int GUARD_ROWS = 128;            // guard rows before and after every destination of op_gemm_ex: one whole row tile each way
constexpr int GUARD_COLS = 32;             // unused columns per row (ldc = N + 32)
constexpr uint32_t GUARD_WORD = 0x7FDA7FDAu;   // NaN as f32, and each half a NaN as f16 and as bf16

// a destination of op_gemm_ex: `live` rows of `cols` elements at row stride cols + GUARD_COLS, between GUARD_ROWS guard rows
struct Guarded {
    DevBuf d; size_t es = 4, ld = 0, live = 0, cols = 0;
    void init(size_t live_rows, size_t n, size_t elem, const float* live_init) {
        es = elem; ld = n + GUARD_COLS; live = live_rows; cols = n;
        std::vector<uint8_t> h(bytes());
        for (size_t i = 0; i + 4 <= h.size(); i += 4) memcpy(&h[i], &GUARD_WORD, 4);
        if (live_init)
            for (size_t r = 0; r < live; ++r) memcpy(&h[((GUARD_ROWS + r) * ld) * es], live_init + r * n, n * 4);
        d.alloc(h.size(), false); h2d_sync(d.p, h.data(), h.size());
    }
    size_t bytes() const { return (2 * GUARD_ROWS + live) * ld * es; }
    void* at() const { return (char*)d.p + GUARD_ROWS * ld * es; }
    // copies the live rows (packed, n elements each) to out and returns how many guard elements differ from the pattern
    long long fetch(void* out) const {
        std::vector<uint8_t> h(bytes());
        NSB_CUDA(cudaMemcpy(h.data(), d.p, h.size(), cudaMemcpyDeviceToHost));
        long long bad = 0;
        for (size_t r = 0; r < 2 * GUARD_ROWS + live; ++r) {
            const bool live_row = r >= GUARD_ROWS && r < GUARD_ROWS + live;
            for (size_t c = live_row ? cols : 0; c < ld; ++c) bad += memcmp(&h[(r * ld + c) * es], &GUARD_WORD, es) != 0;
            if (live_row) memcpy((char*)out + (r - GUARD_ROWS) * cols * es, &h[r * ld * es], cols * es);
        }
        return bad;
    }
};
}  // namespace

long long Engine::op_gemm_ex(const nsb_gemm_op& op, const float* xh, void* y, size_t y_bytes, long long* guard_bad) {
    const Weight& W = op_weight(op.weight);
    const int rows = op.rows, N = W.n_out;
    auto bad = [](const std::string& m) { throw std::invalid_argument("op_gemm_ex: " + m); };
    if (rows < 1) bad("rows must be >= 1");
    if (op.epi < EPI_NONE || op.epi > EPI_PARTIAL) bad("unknown epilogue");
    if (op.out_type < OUT_F32 || op.out_type > OUT_BF16) bad("unknown output type");
    if (op.out_type != OUT_F32 && (op.epi == EPI_RESID || op.epi == EPI_PARTIAL)) bad("residual and split-K outputs are f32");
    if (op.splits < 1 || op.splits > MAX_SPLITS || (op.splits > 1 && op.epi != EPI_PARTIAL)) bad("splits must be 1..8, > 1 only with the split-K epilogue");
    if (op.c0 && op.epi != EPI_PARTIAL) bad("c0 is a split-K destination");
    if (op.c_group < 0 || (op.c_group > 0 && (op.c_drop < 0 || op.c_drop >= op.c_group || rows % op.c_group != 0))) bad("bad output row map");
    if (op.epi == EPI_RESID && !op.c_init) bad("the residual epilogue needs c_init");
    if (strict() && (op.out_type != OUT_F32 || op.epi == EPI_PARTIAL || op.c_group || op.force_bn))
        bad("strict modes run the SIMT / Q8_0 block kernels: f32 output, no split-K, row map or tile config");
    NSB_CUDA(cudaSetDevice(device_));
    const int m_out = op.c_group > 0 ? rows / op.c_group * (op.c_group - op.c_drop) : rows;
    const bool partial = op.epi == EPI_PARTIAL;
    const size_t es = out_elem_size(op.out_type), need = partial ? (size_t)op.splits * m_out * N * 4 : (size_t)m_out * N * es;
    if (y_bytes < need) return -(long long)need;
    ensure_q8s_scratch(rows);
    DevBuf dx, da, dbias;
    const void* A = op_operand(W, xh, rows, dx, da);
    if (op.bias) { dbias.alloc((size_t)N * 4, false); h2d_sync(dbias.p, op.bias, dbias.bytes); }
    // destinations: C (or, split-K, the workspace of the slices that do not go to C0) and C0
    const int ws_planes = partial ? op.splits - (op.c0 ? 1 : 0) : 1;
    Guarded c, c0;
    c.init((size_t)ws_planes * m_out, N, partial ? 4 : es, op.epi == EPI_RESID ? op.c_init : nullptr);
    if (op.c0) c0.init(m_out, N, 4, nullptr);

    GemmArgs g; g.A = A; g.lda = W.n_in; g.W = W.data.p; g.M = rows; g.N = N; g.K = W.n_in; g.bias = op.bias ? dbias.as<float>() : nullptr;
    g.C = c.at(); g.ldc = (long long)c.ld; g.epi = op.epi; g.alpha = op.alpha; g.out_type = op.out_type; g.splits = op.splits;
    g.c_group = op.c_group; g.c_drop = op.c_drop; g.C0 = op.c0 ? c0.at() : nullptr; g.force_bn = op.force_bn; g.force_stages = op.force_stages;
    g.rotate = op.rotate; g.pair = 1;
    if (W.f32) { SplitScratch sc(this, W, rows); gemm_f32w(g, W, false); NSB_CUDA(cudaStreamSynchronize(st_)); }
    else gemm(g, W);
    NSB_CUDA(cudaStreamSynchronize(st_));
    long long nbad = 0;
    if (op.c0) nbad += c0.fetch(y);
    nbad += c.fetch((char*)y + (op.c0 ? (size_t)m_out * N * 4 : 0));
    if (guard_bad) *guard_bad = nbad;
    return N;
}

void Engine::op_layernorm(const float* xh, int rows, const float* planes, int n_planes, float alpha, const float* g1, const float* b1,
                          const float* g2, const float* b2, bool fused, int out_type, float* x_out, void* y) {
    // load_x_reduced folds at most MAX_SPLITS planes: every split-K producer stays within that
    if (rows < 1 || n_planes < 0 || n_planes > MAX_SPLITS || (n_planes && !planes) || !g1 || !b1 || (!g2) != (!b2) || (g2 && !fused))
        throw std::invalid_argument("op_layernorm: bad arguments (rows >= 1, 0..8 planes, g1 / b1, g2 / b2 together and only fused)");
    if (out_type < OUT_F32 || out_type > OUT_BF16) throw std::invalid_argument("op_layernorm: unknown output type");
    NSB_CUDA(cudaSetDevice(device_));
    const size_t n = (size_t)rows * D_MODEL;
    auto up = [](DevBuf& d, const float* h, size_t count) { d.alloc(count * 4, false); h2d_sync(d.p, h, count * 4); };
    DevBuf dx, dp, dg1, db1, dg2, db2, dy;
    up(dx, xh, n); up(dg1, g1, D_MODEL); up(db1, b1, D_MODEL);
    if (n_planes) up(dp, planes, (size_t)n_planes * n);
    if (g2) { up(dg2, g2, D_MODEL); up(db2, b2, D_MODEL); }
    dy.alloc(n * out_elem_size(out_type), false);
    PartialSum ps; ps.part = n_planes ? dp.as<float>() : nullptr; ps.n = n_planes; ps.alpha = alpha;
    if (!fused) launch_layernorm(dx.as<float>(), rows, dg1.as<float>(), db1.as<float>(), dy.p, out_type, ps, st_);
    else launch_layernorm2(dx.as<float>(), rows, dg1.as<float>(), db1.as<float>(), dg2.as<float>(), db2.as<float>(), g2 ? dy.p : nullptr,
                           out_type, ps, st_);
    NSB_CUDA(cudaStreamSynchronize(st_));
    NSB_CUDA(cudaMemcpy(x_out, dx.p, n * 4, cudaMemcpyDeviceToHost));
    if (y && (!fused || g2)) NSB_CUDA(cudaMemcpy(y, dy.p, dy.bytes, cudaMemcpyDeviceToHost));
}

// The step's decode launch (run_decode_kernels / transcribe_full) on the engine's decoder weights, with state, sync buffer and outputs
// of its own. Token and frame buffers are preset to -1 and followed by DEC_GUARD entries holding a pattern the kernel never writes.
void Engine::op_decode(nsb_decode_op& op) {
    constexpr int DEC_GUARD = 4096, MAX_S = 8192;
    constexpr int32_t GUARD_VAL = 0x7FDA7FDA;
    auto bad = [](const std::string& m) { throw std::invalid_argument("op_decode: " + m); };
    const int B = op.B, T = op.T, S = op.S;
    if (B < 1 || B > 1024) bad("B must be 1..1024");
    if (T < 1 || (long long)MAX_SYMBOLS * T > 32767) bad("T must be 1..3276 (the kernel counts emissions in 16 bits)");
    if (S < B || S > MAX_S) bad("S must be B..8192");
    if (!op.slot_of_b || !op.enc_proj || !op.h || !op.c || !op.dec_proj || !op.par || !op.prev_token || !op.cand_valid || !op.tokens ||
        !op.frames || !op.counts) bad("null array");
    NSB_CUDA(cudaSetDevice(device_));
    int sms = 0;
    NSB_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device_));
    if (op.grid != 0 && (op.grid < 2 || op.grid % 2 != 0 || op.grid >= sms)) bad("grid must be 0 or even, 2 <= grid < SM count");
    if (op.pipe_min_n < 0) bad("pipe_min_n must be >= 0");
    std::vector<char> used((size_t)S, 0);
    for (int b = 0; b < B; ++b) {
        const int s = op.slot_of_b[b];
        if (s < 0 || s >= S || used[s]) bad("slot_of_b must hold distinct slots in 0..S-1");
        used[s] = 1;
    }
    for (int s = 0; s < S; ++s) {
        if (op.prev_token[s] < 0 || op.prev_token[s] > BLANK) bad("prev_token must be 0..1024");
        if (op.par[s] != 0 && op.par[s] != 1) bad("par must be 0 or 1");
        if (op.cand_valid[s] != 0 && op.cand_valid[s] != 1) bad("cand_valid must be 0 or 1");
    }

    const size_t n_out = (size_t)B * MAX_SYMBOLS * T, n_tap = (size_t)(MAX_SYMBOLS + 1) * T * VOCAB;
    const size_t st_f = (size_t)S * 4 * HID;
    auto up = [](DevBuf& d, const void* h, size_t bytes) { d.alloc(bytes, false); h2d_sync(d.p, h, bytes); };
    DevBuf d_slot, d_enc, d_h, d_c, d_proj, d_par, d_prev, d_cand, d_tok, d_frm, d_cnt, d_tap, d_tap_n, d_sync;
    up(d_slot, op.slot_of_b, (size_t)B * 4); up(d_enc, op.enc_proj, (size_t)B * T * JOINT * 4);
    up(d_h, op.h, st_f * 4); up(d_c, op.c, st_f * 4); up(d_proj, op.dec_proj, (size_t)S * JOINT * 4);
    up(d_par, op.par, (size_t)S * 4); up(d_prev, op.prev_token, (size_t)S * 4); up(d_cand, op.cand_valid, (size_t)S * 4);
    std::vector<int32_t> preset(n_out + DEC_GUARD, -1);
    std::fill(preset.begin() + n_out, preset.end(), GUARD_VAL);
    up(d_tok, preset.data(), preset.size() * 4); up(d_frm, preset.data(), preset.size() * 4);
    d_cnt.alloc((size_t)B * 4, false); d_tap_n.alloc(4, false); d_sync.alloc(decode_sync_bytes(B), false);
    if (op.logits) {
        const std::vector<float> nan(n_tap, std::numeric_limits<float>::quiet_NaN());
        up(d_tap, nan.data(), n_tap * 4);
    }

    DecodeArgs d{};
    d.w.embed = embed_.as<float>();
    for (int l = 0; l < 2; ++l) { d.w.w_ih[l] = lstm_w_[2 * l].as<float>(); d.w.w_hh[l] = lstm_w_[2 * l + 1].as<float>();
                                  d.w.b_ih[l] = lstm_b_[2 * l].as<float>(); d.w.b_hh[l] = lstm_b_[2 * l + 1].as<float>(); }
    d.w.pred_w = pred_w_.as<float>(); d.w.pred_b = pred_b_.as<float>(); d.w.out_w = jout_w_.as<float>(); d.w.out_b = jout_b_.as<float>();
    d.s.hbuf = d_h.as<float>(); d.s.cbuf = d_c.as<float>(); d.s.par = d_par.as<int>();
    d.s.dec_proj = d_proj.as<float>(); d.s.prev_token = d_prev.as<int>(); d.s.cand_valid = d_cand.as<int>();
    d.enc_proj = d_enc.as<float>(); d.slot_of_b = d_slot.as<int>(); d.B = B; d.T = T;
    d.out_tokens = d_tok.as<int>(); d.out_count = d_cnt.as<int>(); d.out_frames = d_frm.as<int>();
    d.logits_tap = op.logits ? d_tap.as<float>() : nullptr; d.logits_tap_cap = op.logits ? (MAX_SYMBOLS + 1) * T : 0;
    d.logits_tap_n = d_tap_n.as<int>();
    const int used_grid = launch_decode(d, d_sync.p, st_, op.grid, op.pipe_min_n);
    NSB_CUDA(cudaStreamSynchronize(st_));

    auto down = [](void* h, const DevBuf& dv, size_t bytes) { NSB_CUDA(cudaMemcpy(h, dv.p, bytes, cudaMemcpyDeviceToHost)); };
    long long nbad = 0;
    for (const DevBuf* o : {&d_tok, &d_frm}) {
        down(preset.data(), *o, preset.size() * 4);
        for (size_t i = n_out; i < preset.size(); ++i) nbad += preset[i] != GUARD_VAL;
        memcpy(o == &d_tok ? op.tokens : op.frames, preset.data(), n_out * 4);
    }
    down(op.counts, d_cnt, (size_t)B * 4);
    down(op.h, d_h, st_f * 4); down(op.c, d_c, st_f * 4); down(op.dec_proj, d_proj, (size_t)S * JOINT * 4);
    down(op.par, d_par, (size_t)S * 4); down(op.prev_token, d_prev, (size_t)S * 4); down(op.cand_valid, d_cand, (size_t)S * 4);
    int ne = 0;
    down(&ne, d_tap_n, 4);
    op.n_logits = ne;
    if (op.logits) down(op.logits, d_tap, (size_t)std::min(ne, (MAX_SYMBOLS + 1) * T) * VOCAB * 4);
    op.grid_used = used_grid;
    op.guard_bad = nbad;
}

}  // namespace nsb
