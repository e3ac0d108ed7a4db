// gguf_loader.h -- minimal GGUF v3 reader for the nemotron-speech weight layout.
// Replaces the gguf_* / ggml_dup_tensor / fread loop of the reference loader
// (src/nemo-ggml.cpp:83-256); file layout per scripts/convert_to_gguf.py:407-447 and
// docs/TENSOR_SHAPES.md. Tensor bytes are kept exactly as stored (F32 / F16 / Q8_0 / Q4_0).
#pragma once
#include <cstdint>
#include <map>
#include <string>
#include <vector>

namespace nsb {

enum GgmlType : int { GGML_F32 = 0, GGML_F16 = 1, GGML_Q4_0 = 2, GGML_Q8_0 = 8 };

struct GgufTensor {
    std::string name;
    std::vector<int64_t> ne;     // ggml order: ne[0] contiguous
    int type = 0;
    uint64_t offset = 0;         // relative to data section
    size_t nbytes = 0;
    int64_t n_elements() const { int64_t n = 1; for (auto d : ne) n *= d; return n; }
};

struct GgufFile {
    GgufFile() = default;
    GgufFile(const GgufFile&) = delete; GgufFile& operator=(const GgufFile&) = delete;
    ~GgufFile();
    std::string path;
    // the whole file, mapped read-only (open): tensor bytes are consumed straight out of the page cache -- by the host-side
    // dequantisers below and by the engine's chunked asynchronous upload -- never through a per-tensor fopen / fread
    const uint8_t* map = nullptr; size_t map_size = 0;
    const uint8_t* data(const GgufTensor& t) const;     // bounds-checked pointer to the tensor's bytes inside the mapping
    std::map<std::string, uint32_t> u32;      // nemo.* hparams
    std::string vocab_raw;                    // tokenizer.vocab bytes
    std::map<std::string, GgufTensor> tensors;
    uint64_t data_start = 0;

    // Parses header + tensor infos, maps the file, checks that every tensor lies inside it. Throws std::runtime_error with a readable message.
    void open(const std::string& path);
    // Reads the raw bytes of one tensor.
    std::vector<uint8_t> read(const GgufTensor& t) const;
    const GgufTensor& require(const std::string& name) const;
    // Reads a tensor that must be F32 (or F16, widened) into floats.
    std::vector<float> read_f32(const std::string& name) const;
    // Reads any supported tensor as floats: F32 / F16 as stored; Q8_0 blocks (fp16 d + 32 x int8 along ne0) as d * q; Q4_0 blocks
    // (fp16 d + 16 nibble bytes: element i = low nibble of byte i, element i + 16 = high nibble) as d * (q - 8)
    // (scripts/convert_to_gguf.py:93-179; what ggml's dequantize_row_q8_0 / _q4_0 return).
    std::vector<float> read_dequant(const std::string& name) const;
    // 64-bit FNV-1a over the header (metadata and tensor table) and the first and last 4 KiB of every tensor's bytes: tells models
    // apart without a pass over the weights, and does not depend on the file's path
    uint64_t fingerprint() const;
};

// fp16 bits -> float (host)
float half_bits_to_float(uint16_t h);

}  // namespace nsb
