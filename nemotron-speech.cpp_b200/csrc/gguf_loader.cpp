#include "gguf_loader.h"

#include <algorithm>
#include <cstdio>
#include <cmath>
#include <cstring>
#include <stdexcept>

#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>

namespace nsb {

namespace {
struct File {
    FILE* f = nullptr;
    explicit File(const std::string& p) : f(fopen(p.c_str(), "rb")) {}
    ~File() { if (f) fclose(f); }
};
template <class T> T rd(FILE* f) {
    T v{};
    if (fread(&v, sizeof(T), 1, f) != 1) throw std::runtime_error("gguf: unexpected end of file");
    return v;
}
std::string rd_str(FILE* f) {
    uint64_t n = rd<uint64_t>(f);
    if (n > (1ull << 28)) throw std::runtime_error("gguf: string too long");
    std::string s(n, '\0');
    if (n && fread(&s[0], 1, n, f) != n) throw std::runtime_error("gguf: unexpected end of file");
    return s;
}
size_t scalar_size(int t) {
    switch (t) {
        case 0: case 1: case 7: return 1;       // u8 i8 bool
        case 2: case 3: return 2;               // u16 i16
        case 4: case 5: case 6: return 4;       // u32 i32 f32
        case 10: case 11: case 12: return 8;    // u64 i64 f64
        default: return 0;
    }
}
}  // namespace

float half_bits_to_float(uint16_t h) {
    uint32_t sign = (h >> 15) & 1u, exp = (h >> 10) & 0x1fu, man = h & 0x3ffu, f;
    if (exp == 0) {
        float v = ldexpf((float)man, -24);   // zero / subnormal: man * 2^-24, exact
        return sign ? -v : v;
    } else if (exp == 31) f = (sign << 31) | 0x7f800000u | (man << 13);
    else f = (sign << 31) | ((exp + 127 - 15) << 23) | (man << 13);
    float out; memcpy(&out, &f, 4); return out;
}

GgufFile::~GgufFile() { if (map) munmap(const_cast<uint8_t*>(map), map_size); }

const uint8_t* GgufFile::data(const GgufTensor& t) const {
    if (!map || data_start + t.offset + t.nbytes > map_size) throw std::runtime_error("gguf: tensor '" + t.name + "' lies outside the file");
    return map + data_start + t.offset;
}

void GgufFile::open(const std::string& p) {
    path = p;
    File fh(p);
    if (!fh.f) throw std::runtime_error("gguf: cannot open '" + p + "'");
    FILE* f = fh.f;
    char magic[4];
    if (fread(magic, 1, 4, f) != 4 || memcmp(magic, "GGUF", 4) != 0) throw std::runtime_error("gguf: bad magic in '" + p + "'");
    uint32_t version = rd<uint32_t>(f);
    if (version < 2 || version > 3) throw std::runtime_error("gguf: unsupported version " + std::to_string(version));
    int64_t n_tensors = rd<int64_t>(f), n_kv = rd<int64_t>(f);
    if (n_tensors < 0 || n_tensors > (1 << 20) || n_kv < 0 || n_kv > (1 << 20)) throw std::runtime_error("gguf: implausible counts");
    uint64_t alignment = 32;
    for (int64_t i = 0; i < n_kv; ++i) {
        std::string key = rd_str(f);
        int32_t t = rd<int32_t>(f);
        if (t == 8) {
            std::string v = rd_str(f);
            if (key == "tokenizer.vocab") vocab_raw = v;
        } else if (t == 9) {
            int32_t et = rd<int32_t>(f);
            uint64_t n = rd<uint64_t>(f);
            for (uint64_t k = 0; k < n; ++k) {
                if (et == 8) rd_str(f);
                else { size_t sz = scalar_size(et); if (!sz) throw std::runtime_error("gguf: bad array type"); fseek(f, (long)sz, SEEK_CUR); }
            }
        } else {
            size_t sz = scalar_size(t);
            if (!sz) throw std::runtime_error("gguf: unknown kv type " + std::to_string(t));
            uint64_t raw = 0;
            if (fread(&raw, 1, sz, f) != sz) throw std::runtime_error("gguf: unexpected end of file");
            if (t == 4 || t == 5) u32[key] = (uint32_t)raw;
            if (key == "general.alignment") alignment = (uint32_t)raw;
        }
    }
    for (int64_t i = 0; i < n_tensors; ++i) {
        GgufTensor t;
        t.name = rd_str(f);
        uint32_t nd = rd<uint32_t>(f);
        if (nd > 4) throw std::runtime_error("gguf: tensor '" + t.name + "' has >4 dims");
        t.ne.resize(nd);
        for (auto& d : t.ne) d = rd<int64_t>(f);
        t.type = rd<int32_t>(f);
        t.offset = rd<uint64_t>(f);
        int64_t n = t.n_elements();
        switch (t.type) {
            case GGML_F32: t.nbytes = (size_t)n * 4; break;
            case GGML_F16: t.nbytes = (size_t)n * 2; break;
            case GGML_Q8_0:
                if (t.ne.empty() || t.ne[0] % 32) throw std::runtime_error("gguf: Q8_0 tensor '" + t.name + "' ne0 % 32 != 0");
                t.nbytes = (size_t)n / 32 * 34; break;
            case GGML_Q4_0:
                if (t.ne.empty() || t.ne[0] % 32) throw std::runtime_error("gguf: Q4_0 tensor '" + t.name + "' ne0 % 32 != 0");
                t.nbytes = (size_t)n / 32 * 18; break;
            default: throw std::runtime_error("gguf: tensor '" + t.name + "' has unsupported type " + std::to_string(t.type) +
                                              " (supported: F32, F16, Q8_0, Q4_0)");
        }
        tensors[t.name] = t;
    }
    uint64_t pos = (uint64_t)ftell(f);
    data_start = (pos + alignment - 1) / alignment * alignment;
    // map the file and make sure every tensor is inside it (a truncated download fails here, by name, not in the middle of a load)
    const int fd = ::open(p.c_str(), O_RDONLY);
    struct stat sb;
    if (fd < 0 || fstat(fd, &sb) != 0) { if (fd >= 0) ::close(fd); throw std::runtime_error("gguf: cannot open '" + p + "'"); }
    map_size = (size_t)sb.st_size;
    void* m = map_size ? mmap(nullptr, map_size, PROT_READ, MAP_PRIVATE, fd, 0) : MAP_FAILED;
    ::close(fd);
    if (m == MAP_FAILED) { map_size = 0; throw std::runtime_error("gguf: cannot map '" + p + "'"); }
    map = (const uint8_t*)m;
    madvise(m, map_size, MADV_SEQUENTIAL);
    for (const auto& kv : tensors) {
        const GgufTensor& t = kv.second;
        if (t.offset % alignment != 0) throw std::runtime_error("gguf: tensor '" + t.name + "' is not aligned to " + std::to_string(alignment) + " bytes");
        if (data_start + t.offset + t.nbytes > map_size)
            throw std::runtime_error("gguf: file truncated: tensor '" + t.name + "' needs bytes up to " + std::to_string(data_start + t.offset + t.nbytes) +
                                     " but the file has " + std::to_string(map_size));
    }
}

const GgufTensor& GgufFile::require(const std::string& name) const {
    auto it = tensors.find(name);
    if (it == tensors.end()) throw std::runtime_error("gguf: missing tensor: " + name);
    return it->second;
}

std::vector<uint8_t> GgufFile::read(const GgufTensor& t) const {
    const uint8_t* p = data(t);
    return std::vector<uint8_t>(p, p + t.nbytes);
}

std::vector<float> GgufFile::read_f32(const std::string& name) const {
    const GgufTensor& t = require(name);
    std::vector<uint8_t> raw = read(t);
    std::vector<float> out((size_t)t.n_elements());
    if (t.type == GGML_F32) memcpy(out.data(), raw.data(), raw.size());
    else if (t.type == GGML_F16) for (size_t i = 0; i < out.size(); ++i) { uint16_t h; memcpy(&h, &raw[2 * i], 2); out[i] = half_bits_to_float(h); }
    else throw std::runtime_error("gguf: tensor '" + name + "' expected F32/F16");
    return out;
}

std::vector<float> GgufFile::read_dequant(const std::string& name) const {
    const GgufTensor& t = require(name);
    std::vector<uint8_t> raw = read(t);
    std::vector<float> out((size_t)t.n_elements());
    if (t.type == GGML_F32) memcpy(out.data(), raw.data(), raw.size());
    else if (t.type == GGML_F16) { for (size_t i = 0; i < out.size(); ++i) { uint16_t h; memcpy(&h, &raw[2 * i], 2); out[i] = half_bits_to_float(h); } }
    else if (t.type == GGML_Q8_0) {                       // block = fp16 d + 32 x int8 along ne0 (convert_to_gguf.py:93-129)
        const size_t nb = out.size() / 32;
        for (size_t b = 0; b < nb; ++b) {
            uint16_t h; memcpy(&h, &raw[b * 34], 2); const float d = half_bits_to_float(h);
            const int8_t* q = (const int8_t*)&raw[b * 34 + 2];
            for (int i = 0; i < 32; ++i) out[b * 32 + i] = d * (float)q[i];
        }
    } else if (t.type == GGML_Q4_0) {                     // block = fp16 d + 16 nibble bytes: element i = low nibble of byte i, i + 16 = high nibble;
        const size_t nb = out.size() / 32;                // value = d * (q - 8) (convert_to_gguf.py:132-179)
        for (size_t b = 0; b < nb; ++b) {
            uint16_t h; memcpy(&h, &raw[b * 18], 2); const float d = half_bits_to_float(h);
            const uint8_t* q = &raw[b * 18 + 2];
            for (int i = 0; i < 16; ++i) { out[b * 32 + i] = d * (float)((int)(q[i] & 0x0F) - 8); out[b * 32 + 16 + i] = d * (float)((int)(q[i] >> 4) - 8); }
        }
    } else throw std::runtime_error("unsupported tensor type for " + name);
    return out;
}

uint64_t GgufFile::fingerprint() const {
    uint64_t h = 0xcbf29ce484222325ull;
    auto eat = [&](const uint8_t* p, size_t n) { for (size_t i = 0; i < n; ++i) { h ^= p[i]; h *= 0x100000001b3ull; } };
    eat(map, (size_t)std::min<uint64_t>(data_start, map_size));   // magic, metadata, tensor table
    for (const auto& kv : tensors) {                               // name order
        const GgufTensor& t = kv.second;
        const uint8_t* p = data(t);
        const size_t edge = std::min<size_t>(t.nbytes, 4096);
        eat(p, edge);
        eat(p + t.nbytes - edge, edge);
    }
    return h;
}

}  // namespace nsb
