// stream_state.cu -- stream snapshots: nsb_stream_export / nsb_stream_import (include/nsb200.h). A snapshot holds everything that
// decides a stream's future output -- the slot's device state and its host bookkeeping -- so that a stream can be suspended, resumed
// in another engine, or moved between GPUs. Layout, compatibility rule and checksum: DESIGN.md §11.
//
//   header (SnapHeader, 152 bytes) | K/V ring | conv state | mel history | dec_h | dec_c | dec_proj | PCM (pad 8) | tokens (pad 8) | checksum
//
// Every section starts at an 8-byte boundary; integers are little-endian. checksum = sum over the blob's u64 words w_i (i from 0, the
// checksum word excluded) of mix(w_i + (i + 1) * 0x9E3779B97F4A7C15) mod 2^64, mix = the splitmix64 finalizer. Being a sum, the bulk
// sections are hashed on the device where they already are (export) or have just been copied to (import), the rest on the host.
#include "engine.h"

#include <algorithm>
#include <cstring>

namespace nsb {

namespace {

constexpr char SNAP_MAGIC[4] = {'N', 'S', 'B', 'S'};
constexpr uint32_t SNAP_VERSION = 1;
constexpr uint64_t SNAP_GOLDEN = 0x9E3779B97F4A7C15ull;

struct SnapHeader {
    char magic[4]; uint32_t version;
    uint64_t total_bytes, fingerprint;
    int64_t n_layers, R, kv_dtype, compute;                                   // must match the importing engine
    int64_t ring_pos, valid_len, cc_par, dec_par, prev_token, cand_valid;     // the slot's device scalars
    int64_t base, n_pushed, chunk_idx, chunks_done, n_pcm, n_tokens;          // HostStream
};
static_assert(sizeof(SnapHeader) == 152, "snapshot header layout");

__host__ __device__ inline uint64_t snap_mix(uint64_t z) {
    z ^= z >> 30; z *= 0xBF58476D1CE4E5B9ull;
    z ^= z >> 27; z *= 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

uint64_t host_checksum(const uint8_t* p, size_t bytes, size_t first_word) {
    uint64_t s = 0;
    for (size_t i = 0; i < bytes / 8; ++i) { uint64_t w; memcpy(&w, p + 8 * i, 8); s += snap_mix(w + (first_word + i + 1) * SNAP_GOLDEN); }
    return s;
}

struct SnapSegs { const uint64_t* p[SNAP_BULK]; unsigned long long words[SNAP_BULK], first[SNAP_BULK]; };

__global__ void __launch_bounds__(256) snapshot_checksum_kernel(SnapSegs t, unsigned long long* out) {
    unsigned long long acc = 0;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
#pragma unroll 1
    for (int k = 0; k < SNAP_BULK; ++k)
        for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < t.words[k]; i += stride)
            acc += snap_mix(__ldg(t.p[k] + i) + (t.first[k] + i + 1) * SNAP_GOLDEN);
    for (int o = 16; o; o >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0) atomicAdd(out, acc);                         // a sum mod 2^64: the order does not matter
}

size_t pad8(size_t n) { return (n + 7) & ~(size_t)7; }

}  // namespace

size_t Engine::snapshot_sections(int s, void** ptr, size_t* bytes) const {
    const size_t kvb = (size_t)n_layers * 2 * (ATT_L + T) * D_MODEL * kv_elem_size(kv_dtype);
    const size_t cb = (size_t)2 * n_layers * (CONV_K - 1) * D_MODEL * 4, mb = (size_t)PRE_CACHE * N_MELS * 4, db = (size_t)4 * HID * 4;
    const size_t b[SNAP_BULK] = {kvb, cb, mb, db, db, (size_t)JOINT * 4};
    const DevBuf* buf[SNAP_BULK] = {&kv_, &conv_cache_, &mel_hist_, &dec_h_, &dec_c_, &dec_proj_};
    size_t total = 0;
    for (int k = 0; k < SNAP_BULK; ++k) { ptr[k] = (char*)buf[k]->p + (size_t)s * b[k]; bytes[k] = b[k]; total += b[k]; }
    return total;
}

uint64_t Engine::device_checksum(void* const* ptr, const size_t* bytes, size_t first_word) {
    if (!snap_sum_.p) snap_sum_.alloc(8);
    SnapSegs t;
    for (int k = 0; k < SNAP_BULK; ++k) { t.p[k] = (const uint64_t*)ptr[k]; t.words[k] = bytes[k] / 8; t.first[k] = first_word; first_word += bytes[k] / 8; }
    NSB_CUDA(cudaMemsetAsync(snap_sum_.p, 0, 8, st_));
    snapshot_checksum_kernel<<<148 * 4, 256, 0, st_>>>(t, snap_sum_.as<unsigned long long>());
    NSB_CUDA(cudaGetLastError());
    count_launch();
    uint64_t sum = 0;
    NSB_CUDA(cudaMemcpyAsync(&sum, snap_sum_.p, 8, cudaMemcpyDeviceToHost, st_));
    NSB_CUDA(cudaStreamSynchronize(st_));
    return sum;
}

long long Engine::export_stream(int s, void* out, size_t cap) {
    collect_all();                                                            // tokens of the steps in flight join the queue
    if (s < 0 || s >= max_streams || !hs_[s].open) throw std::invalid_argument("nsb_stream_export: stream " + std::to_string(s) + " is not open");
    const HostStream& h = hs_[s];
    void* ptr[SNAP_BULK]; size_t bytes[SNAP_BULK];
    const size_t bulk = snapshot_sections(s, ptr, bytes);
    const size_t n_pcm = h.buf.size() - h.head, n_tok = h.tokens.size();
    const size_t pcm_off = sizeof(SnapHeader) + bulk, tok_off = pcm_off + pad8(n_pcm * 2), sum_off = tok_off + pad8(n_tok * 4);
    const size_t total = sum_off + 8;
    if (!out) return (long long)total;
    if (cap < total) throw std::invalid_argument("nsb_stream_export: buffer of " + std::to_string(cap) + " bytes, the snapshot needs " + std::to_string(total));
    NSB_CUDA(cudaSetDevice(device_));
    join_decode_stream();                                                     // decoder state of the slot: no decode may still be running
    uint8_t* o = (uint8_t*)out;
    int sc[6];
    int* const src[6] = {ring_pos_.as<int>(), valid_len_.as<int>(), cc_par_.as<int>(), dec_par_.as<int>(), prev_token_.as<int>(), cand_valid_.as<int>()};
    for (int k = 0; k < 6; ++k) NSB_CUDA(cudaMemcpyAsync(&sc[k], src[k] + s, 4, cudaMemcpyDeviceToHost, st_));
    size_t off = sizeof(SnapHeader);
    for (int k = 0; k < SNAP_BULK; ++k) { NSB_CUDA(cudaMemcpyAsync(o + off, ptr[k], bytes[k], cudaMemcpyDeviceToHost, st_)); off += bytes[k]; }
    uint64_t sum = device_checksum(ptr, bytes, sizeof(SnapHeader) / 8);      // synchronises st_: the copies above have landed

    SnapHeader hd{};
    memcpy(hd.magic, SNAP_MAGIC, 4); hd.version = SNAP_VERSION;
    hd.total_bytes = total; hd.fingerprint = fingerprint;
    hd.n_layers = n_layers; hd.R = R; hd.kv_dtype = kv_dtype; hd.compute = compute;
    hd.ring_pos = sc[0]; hd.valid_len = sc[1]; hd.cc_par = sc[2]; hd.dec_par = sc[3]; hd.prev_token = sc[4]; hd.cand_valid = sc[5];
    hd.base = h.base; hd.n_pushed = h.n_pushed; hd.chunk_idx = h.chunk_idx; hd.chunks_done = h.chunks_done;
    hd.n_pcm = (int64_t)n_pcm; hd.n_tokens = (int64_t)n_tok;
    memcpy(o, &hd, sizeof hd);
    memset(o + pcm_off, 0, sum_off - pcm_off);                                // padding
    if (n_pcm) memcpy(o + pcm_off, h.buf.data() + h.head, n_pcm * 2);
    int32_t* tk = reinterpret_cast<int32_t*>(o + tok_off);
    for (size_t i = 0; i < n_tok; ++i) { const int32_t v = h.tokens[i]; memcpy(tk + i, &v, 4); }
    sum += host_checksum(o, sizeof hd, 0) + host_checksum(o + pcm_off, sum_off - pcm_off, pcm_off / 8);
    memcpy(o + sum_off, &sum, 8);
    return (long long)total;
}

int Engine::import_stream(const void* blob, size_t nbytes) {
    collect_all();
    const uint8_t* b = (const uint8_t*)blob;
    const std::string at = "nsb_stream_import: ";
    if (nbytes < sizeof(SnapHeader) + 8) throw FormatError(at + "size: " + std::to_string(nbytes) + " bytes is shorter than a snapshot header");
    SnapHeader hd; memcpy(&hd, b, sizeof hd);
    if (memcmp(hd.magic, SNAP_MAGIC, 4) != 0) throw FormatError(at + "magic: not a stream snapshot");
    if (hd.version != SNAP_VERSION) throw FormatError(at + "version: format version " + std::to_string(hd.version) + ", this library reads " + std::to_string(SNAP_VERSION));
    if (hd.total_bytes != nbytes) throw FormatError(at + "size: the header says " + std::to_string(hd.total_bytes) + " bytes, the buffer has " + std::to_string(nbytes));
    auto need = [&](bool ok, const char* field) { if (!ok) throw FormatError(at + field + " out of range"); };
    need(hd.n_layers >= 1 && hd.n_layers <= 4096, "n_layers");
    need(hd.R >= 0 && hd.R <= 64, "att_right_context");
    need(hd.kv_dtype >= 0 && hd.kv_dtype <= 2, "kv_dtype");
    need(hd.compute >= NSB_COMPUTE_F32 && hd.compute <= NSB_COMPUTE_Q8_0_STRICT, "compute");
    need(hd.n_pcm >= 0 && (uint64_t)hd.n_pcm <= nbytes / 2, "n_pcm");
    need(hd.n_tokens >= 0 && (uint64_t)hd.n_tokens <= nbytes / 4, "n_tokens");
    // section lengths: the layout the header's own geometry implies must fill the buffer exactly
    const int64_t hT = 1 + hd.R, hCap = ATT_L + hT;
    const size_t hbulk = (size_t)hd.n_layers * 2 * hCap * D_MODEL * kv_elem_size((int)hd.kv_dtype) + (size_t)2 * hd.n_layers * (CONV_K - 1) * D_MODEL * 4 +
                         (size_t)PRE_CACHE * N_MELS * 4 + (size_t)2 * 4 * HID * 4 + (size_t)JOINT * 4;
    const size_t pcm_off = sizeof(SnapHeader) + hbulk, tok_off = pcm_off + pad8((size_t)hd.n_pcm * 2), sum_off = tok_off + pad8((size_t)hd.n_tokens * 4);
    if (sum_off + 8 != nbytes) throw FormatError(at + "size: section lengths (n_layers, att_right_context, kv_dtype, n_pcm, n_tokens) do not add up to " + std::to_string(nbytes) + " bytes");
    // the engine must run the same state geometry
    auto fit = [&](int64_t snap, int64_t eng, const char* field) {
        if (snap != eng) throw std::invalid_argument(at + field + " of the snapshot is " + std::to_string(snap) + ", the engine's is " + std::to_string(eng));
    };
    fit(hd.n_layers, n_layers, "n_layers"); fit(hd.R, R, "att_right_context"); fit(hd.kv_dtype, kv_dtype, "kv_dtype");
    // the scalars index the ring, the conv parities, the vocabulary and the host PCM: each in the range the kernels / host code produce
    need(hd.ring_pos >= 0 && hd.ring_pos < ATT_L + T, "ring_pos");
    need(hd.valid_len >= 0 && hd.valid_len <= ATT_L, "valid_len");
    need(hd.cc_par == 0 || hd.cc_par == 1, "cc_par");
    need(hd.dec_par == 0 || hd.dec_par == 1, "dec_par");
    need(hd.prev_token >= 0 && hd.prev_token <= BLANK, "prev_token");
    need(hd.cand_valid == 0 || hd.cand_valid == 1, "cand_valid");
    need(hd.chunk_idx >= 0 && hd.chunk_idx <= (1ll << 40), "chunk_idx");
    need(hd.chunks_done == hd.chunk_idx, "chunks_done");
    need(hd.base == std::max(0ll, 8ll * T * HS_HOP * hd.chunk_idx - HS_NFFT / 2 - 1), "base");   // what hs_launched keeps
    need(hd.n_pushed - hd.base == hd.n_pcm, "n_pushed");
    std::vector<int32_t> toks((size_t)hd.n_tokens);
    if (!toks.empty()) memcpy(toks.data(), b + tok_off, toks.size() * 4);
    for (int32_t t : toks) need(t >= 0 && t < BLANK, "token id");

    int slot = -1;
    for (int s = 0; s < max_streams && slot < 0; ++s) if (!hs_[s].open) slot = s;
    if (slot < 0) throw std::runtime_error("no free stream slot (max_streams = " + std::to_string(max_streams) + ")");
    NSB_CUDA(cudaSetDevice(device_));
    join_decode_stream();
    // the slot is free: whatever lands in it stays unused unless every check below passes (the next open re-zeroes it)
    void* ptr[SNAP_BULK]; size_t bytes[SNAP_BULK];
    snapshot_sections(slot, ptr, bytes);
    size_t off = sizeof(SnapHeader);
    for (int k = 0; k < SNAP_BULK; ++k) { NSB_CUDA(cudaMemcpyAsync(ptr[k], b + off, bytes[k], cudaMemcpyHostToDevice, st_)); off += bytes[k]; }
    uint64_t sum = device_checksum(ptr, bytes, sizeof(SnapHeader) / 8);
    sum += host_checksum(b, sizeof hd, 0) + host_checksum(b + pcm_off, sum_off - pcm_off, pcm_off / 8);
    uint64_t stored; memcpy(&stored, b + sum_off, 8);
    if (sum != stored) throw FormatError(at + "checksum mismatch: the snapshot is corrupted");
    fit(hd.compute, compute, "compute");
    if (hd.fingerprint != fingerprint) throw std::invalid_argument(at + "model fingerprint differs: the snapshot comes from another model file");

    const int sc[6] = {(int)hd.ring_pos, (int)hd.valid_len, (int)hd.cc_par, (int)hd.dec_par, (int)hd.prev_token, (int)hd.cand_valid};
    int* const dst[6] = {ring_pos_.as<int>(), valid_len_.as<int>(), cc_par_.as<int>(), dec_par_.as<int>(), prev_token_.as<int>(), cand_valid_.as<int>()};
    for (int k = 0; k < 6; ++k) NSB_CUDA(cudaMemcpyAsync(dst[k] + slot, &sc[k], 4, cudaMemcpyHostToDevice, st_));
    NSB_CUDA(cudaStreamSynchronize(st_));
    HostStream& h = hs_[slot];
    hs_clear(h);
    h.buf.resize((size_t)hd.n_pcm);
    if (hd.n_pcm) memcpy(h.buf.data(), b + pcm_off, (size_t)hd.n_pcm * 2);
    h.base = hd.base; h.n_pushed = hd.n_pushed; h.chunk_idx = hd.chunk_idx; h.chunks_done = hd.chunks_done;
    h.tokens.assign(toks.begin(), toks.end());
    h.open = true;
    return slot;
}

}  // namespace nsb
