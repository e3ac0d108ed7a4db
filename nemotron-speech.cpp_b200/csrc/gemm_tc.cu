// gemm_tc.cu -- tcgen05 / TMEM / TMA GEMM for sm_100a:  C[M,N] = A[M,K] * W[N,K]^T  (fp16 / bf16 / tf32 operands, fp32 accumulate)
//
// This is the kernel behind every per-layer weight matrix of the FastConformer block (FFN linear1/2, fused QKV,
// attention out, conv pointwise 1/2) when the engine computes in F16 / BF16 / Q8_0 mode, i.e. what the reference
// delegates to ggml_mul_mat (src/nemo-stream.cpp:457-459, :542, :571-573, :626, :649).
//
// Structure (one CTA = one 128 x BN output tile, 192 threads, warp-specialised):
//   warp 0   : TMA producer   -- cp.async.bulk.tensor.2d of the A tile [128 x 64] and the W tile [BN x 64] per k-block
//                                into a STAGES-deep shared-memory ring (128-byte swizzle), completion on mbarriers
//   warp 1   : MMA issuer     -- one elected lane issues tcgen05.mma.cta_group::1.kind::f16 (M=128, N=BN, K=16) x4 per
//                                k-block, accumulating in TMEM; tcgen05.commit releases the smem stage / signals the epilogue
//   warps 2-5: epilogue       -- tcgen05.ld the fp32 accumulator (each warp owns the TMEM lane quarter warp_id % 4),
//                                apply bias / SiLU / residual and store (f32 or 16-bit)
// Both operands are K-major, so the same shared-memory descriptor recipe serves A and W.
// EB = 4 instantiates the same pipeline for fp32 operands as kind::tf32 (32 elements per 128-byte swizzle row, K = 8 per
// MMA; TMA rounds fp32 -> tf32 on load): used by the 16-bit / Q8_0 engine modes for the matrices every GGUF keeps in F32
// (subsampling 1x1 convs and out-projection = the implicit-GEMM half of the dw-striding stem, joint.enc).
// Rows of A beyond M are zero-filled by TMA (tensor map extent = M), so small batches need no padding.
#include <cuda.h>

#include <algorithm>
#include <initializer_list>
#include <mutex>
#include <stdexcept>
#include <string>

#include "kernels.cuh"

namespace nsb {

NSB_DEFINE_TRACE_BINDER(trace_bind_gemm_tc)

bool pair_gemm_enabled() {
    static const bool on = [] { const char* e = getenv("NSB_PAIR_GEMM"); return !(e && e[0] == '0'); }();
    return on;
}

// NSB_Q8_PAIR=1: Q8_0 / Q4_0 dequantisation fused into the 256-row CTA-pair tiles at large batches (gemm_q8_pair256_kernel). Off by
// default: measured 7.55 ms per 256-stream x 560 ms step against 6.79 ms for the layer-ahead fp16 shadows (which run at exactly the bf16
// engine's speed: 6.78 ms) -- the dequantise -> relay -> MMA chain lengthens every stage's turnaround and three stages are all that fit
// next to a second CTA. Read per launch, so a test can switch it between engines of one process.
bool q8_pair256_enabled() {
    const char* e = getenv("NSB_Q8_PAIR");
    return e && e[0] == '1';
}

static bool pair256_enabled() {
    static const bool on = [] { const char* e = getenv("NSB_PAIR256"); return !(e && e[0] == '0'); }();
    return on;
}

// persistent variant of the 256-row pair tiles (two TMEM accumulators, one ring across tiles): NSB_PAIR256_PERSIST=0/1, read per launch
// (launches happen at graph capture, not at replay) so that a test can switch it between engines of one process
static bool pair256_persist_enabled() {
    const char* e = getenv("NSB_PAIR256_PERSIST");
    return e ? e[0] == '1' : false;
}

static int pair256_min_tiles() {
    static const int v = [] { const char* e = getenv("NSB_PAIR256_MIN_TILES"); return e ? atoi(e) : 4; }();
    return v;
}

namespace {

constexpr int BM = 128, ROW_BYTES = 128, UMMA_K_BYTES = 32;      // one k-block = one 128-byte swizzle row per tile row; 4 MMAs per k-block
constexpr int TC_THREADS = 192;
constexpr int Q8_THREADS = 320, Q8_DEQ = 256;
constexpr int QP_THREADS = 192, QP_DEQ = 128;                   // Q8_0 pair-tile kernel: warps 2-5 dequantise, then run the epilogue (two CTAs per SM)                    // Q8_0 kernel: warps 2-9 dequantise (warps 2-5 also run the epilogue)

// ------------------------------------------------------------------ PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// bounded wait: a protocol bug traps instead of hanging the GPU
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    const uint32_t addr = smem_u32(bar);
    for (uint32_t it = 0; it < (1u << 26); ++it) {
        uint32_t done;
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done) : "r"(addr), "r"(parity) : "memory");
        if (done) return;
    }
    __trap();
}
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* tm, uint64_t* bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(tm), "r"(smem_u32(bar)), "r"(c0), "r"(c1) : "memory");
}
// L2 prefetch of one tensor-map box (no shared-memory destination, no barrier): used before the dependency wait to start
// HBM -> L2 streaming of the part of the weight slab that does not fit the shared-memory ring yet
__device__ __forceinline__ void tma_prefetch_2d(const CUtensorMap* tm, int c0, int c1) {
    asm volatile("cp.async.bulk.prefetch.tensor.2d.L2.global [%0, {%1, %2}];" ::"l"(tm), "r"(c0), "r"(c1) : "memory");
}
// ---- thread-block clusters: A-tile multicast (every CTA of a cluster row needs the same activation tile) ----
__device__ __forceinline__ uint32_t cluster_ctarank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void tma_load_2d_mc(void* smem_dst, const CUtensorMap* tm, uint64_t* bar, int c0, int c1, uint16_t mask) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%3, %4}], [%2], %5;"
        ::"r"(smem_u32(smem_dst)), "l"(tm), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "h"(mask) : "memory");
}
__device__ __forceinline__ void umma_commit_mc(uint64_t* bar, uint16_t mask) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(smem_u32(bar)), "h"(mask) : "memory");
}
// ---- CTA pair (cta_group::2): one MMA spans two SMs; each CTA stages its half of both operands ----
__device__ __forceinline__ void tma_load_2d_pair(void* smem_dst, const CUtensorMap* tm, uint64_t* bar, int c0, int c1) {
    // executed by both CTAs; the peer bit of the barrier address is cleared so that the bytes are counted on CTA 0's barrier
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4}], [%2], %5;"
        ::"r"(smem_u32(smem_dst)), "l"(tm), "r"(smem_u32(bar) & 0xFEFFFFFFu), "r"(c0), "r"(c1), "l"(0x1000000000000000ull) : "memory");
}
__device__ __forceinline__ void umma_f16_pair(uint32_t tmem_c, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_c), "l"(da), "l"(db), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_commit_pair(uint64_t* bar) {          // arrives on the barrier at this offset in BOTH CTAs
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(smem_u32(bar)), "h"((uint16_t)3) : "memory");
}
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* slot, uint32_t cols) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "r"(cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t addr, uint32_t cols) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(cols) : "memory");
}
__device__ __forceinline__ void tmem_alloc(uint32_t* slot, uint32_t cols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "r"(cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t addr, uint32_t cols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(cols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void umma_f16(uint32_t tmem_c, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_c), "l"(da), "l"(db), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_tf32(uint32_t tmem_c, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_c), "l"(da), "l"(db), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
        "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
          "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]),
          "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]),
          "=r"(r[30]), "=r"(r[31])
        : "r"(taddr) : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}

// K-major, SWIZZLE_128B shared-memory matrix descriptor (cute::UMMA::SmemDescriptor): 8-row atoms of 1024 B,
// SBO = 1024 B between atoms, LBO unused for swizzled K-major (encoded 1), version = 1, layout_type = 2.
__device__ __forceinline__ uint64_t make_desc(uint32_t smem_addr) {
    return (uint64_t)((smem_addr >> 4) & 0x3FFF) | ((uint64_t)1 << 16) | ((uint64_t)(1024 >> 4) << 32) | ((uint64_t)1 << 46) |
           ((uint64_t)2 << 61);
}
// cute::UMMA::InstrDescriptor: c=F32, a/b = F16 (0) / BF16 (1) for kind::f16, TF32 (2) for kind::tf32; K-major both, N>>3 @17, M>>4 @24
__host__ __device__ constexpr uint32_t make_idesc(int fmt /*0 f16, 1 bf16, 2 tf32*/, int n, int m = BM) {
    return (1u << 4) | ((uint32_t)fmt << 7) | ((uint32_t)fmt << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}
// TMEM allocations are powers of two >= 32 columns
__host__ __device__ constexpr uint32_t tmem_cols_for(int n) { return n <= 32 ? 32u : n <= 64 ? 64u : n <= 128 ? 128u : n <= 256 ? 256u : 512u; }

struct TcParams {
    int M, N, K;
    const float* bias; void* C; long long ldc; int epi; float alpha; int out_type; int fmt; int rot;
    int c_group, c_drop;       // output row map: row r -> (r / c_group) * (c_group - c_drop) + r % c_group - c_drop, rows with r % c_group < c_drop are dropped
    void* C0; int m_out;       // EPI_PARTIAL: slice 0 (+bias) goes to C0 when set, slices z >= 1 to C + (z-1) * m_out * ldc
    int w_dyn = 0;             // W is produced by the previous kernel (Q8_0 weights dequantised once per launch): no weight TMA before the dependency wait
    int a_fold = 0;            // 3xTF32 (kind::tf32 only): W holds [hi | lo | hi] along K' = 3 a_fold, A holds [hi | lo] (2 a_fold columns):
                               // the A column of k index kc is kc (kc < a_fold) or kc - a_fold
};

// Epilogue of one 128 x BN tile (4 warps; TMEM lane quarter = warp % 4): tcgen05.ld the fp32 accumulator, apply the fused
// epilogue, store. Called by warps 2-5 after the accumulator barrier.
//
// tcgen05.ld hands thread l of a warp ROW l of the tile (32 consecutive columns per step). Stored that way a warp-wide
// st.global.v4 touches 32 different rows = 32 separate 16-byte pieces per instruction, and at large batches the epilogue, not the
// main loop, set the GEMM's pace (profiles/r01_notes.md). So each 32 x 32 chunk is transposed through a warp-private shared-memory
// patch (row stride 36 floats: conflict-free both ways): 8 lanes then cover 128 contiguous bytes of one output row, 4 rows per
// instruction. The patch lives in the first pipeline stages of the A ring, which are idle once the accumulator barrier has fired
// (every TMA write landed, every MMA read retired).
constexpr int EPI_RS = 36;                                       // floats per staged row
constexpr int EPI_STAGE_BYTES = 4 * 32 * EPI_RS * 4;             // 4 epilogue warps

// row0 = global output row of lane 0 of this warp (its TMEM lanes are (warp % 4) * 32 ..), n0 = global column of TMEM column 0,
// BN = number of accumulator columns this warp reads, stage = this CTA's staging area (EPI_STAGE_BYTES, 16-byte aligned)
// parity / zs: phase of the accumulator barrier and k-slice of the tile (persistent kernel: several tiles per CTA; otherwise 0 / blockIdx.z)
template <int BN>
__device__ __forceinline__ void tc_epilogue_at(const TcParams& p, uint32_t tmem_base, uint64_t* tmem_full, int warp, int row0, int n0, int trace_slot,
                                               uint8_t* stage_base, uint32_t parity = 0, int zs = -1) {
        const int zslice = zs >= 0 ? zs : (int)blockIdx.z;
        const bool tracer = trace_slot >= 0 && threadIdx.x == 64;
        const int q = warp & 3, lane = threadIdx.x & 31;
        float* stage = reinterpret_cast<float*>(stage_base) + q * 32 * EPI_RS;
        const int r4 = lane >> 3, c4 = (lane & 7) * 4;          // transposed mapping: pass i covers rows 4 i + r4, this lane columns c4 .. c4 + 3
        // output rows of this lane's 8 passes (-1 = dropped / beyond M)
        int orow[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int row = row0 + 4 * i + r4;
            int o = row; bool live = row < p.M;
            if (p.c_group > 0) { const int rr = row % p.c_group; o = (row / p.c_group) * (p.c_group - p.c_drop) + rr - p.c_drop; live = live && rr >= p.c_drop; }
            orow[i] = live ? o : -1;
        }
        float* part_base = nullptr;
        if (p.epi == EPI_PARTIAL)
            part_base = p.C0 ? (zslice == 0 ? (float*)p.C0 : (float*)p.C + (size_t)(zslice - 1) * p.m_out * p.ldc)
                             : (float*)p.C + (size_t)zslice * p.m_out * p.ldc;
        const bool add_bias = p.bias && (p.epi != EPI_PARTIAL || zslice == 0);
        const bool out16 = p.epi != EPI_PARTIAL && p.epi != EPI_RESID && p.out_type != OUT_F32;
        int orow_own = -1;                                      // output row of this thread's own TMEM lane (16-bit path)
        {
            const int row = row0 + lane;
            int o = row; bool live = row < p.M;
            if (p.c_group > 0) { const int rr = row % p.c_group; o = (row / p.c_group) * (p.c_group - p.c_drop) + rr - p.c_drop; live = live && rr >= p.c_drop; }
            if (live) orow_own = o;
        }
        pdl_wait();                                             // C / bias may be produced (or still read) by the previous kernel
        if (tracer) trace_mark(trace_slot, 2);
        mbar_wait(tmem_full, parity);
        tc_fence_after();
        if (tracer) trace_mark(trace_slot, 3);
#pragma unroll 1
        for (int c = 0; c < BN; c += 32) {
            // columns of this chunk inside the tile and the matrix: 32, or 16 when BN is an odd multiple of 16 / the last tile overhangs N
            const int nv = min(32, min(BN - c, p.N - (n0 + c)));
            if (nv <= 0) break;                                 // warp-uniform
            uint32_t r[32];
            tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)c, r);
            const int n = n0 + c;
            float v[32];
#pragma unroll
            for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
            if (add_bias) {
#pragma unroll
                for (int i = 0; i < 32; ++i) if (i < nv) v[i] += p.bias[n + i];
            }
            if (p.epi == EPI_SILU) {                            // result is rounded to 16 bits: MUFU-based exp / reciprocal is exact enough
#pragma unroll
                for (int i = 0; i < 32; ++i) v[i] = silu_f(v[i]);
            } else if (p.epi == EPI_RELU) {
#pragma unroll
                for (int i = 0; i < 32; ++i) v[i] = fmaxf(v[i], 0.f);
            }
            if (out16) {
                // 16-bit results: a thread's 32 columns are 64 contiguous bytes = two full sectors; stored straight from the row-per-thread
                // layout (the transpose below costs more shared-memory traffic than it saves here: measured, profiles/r01_notes.md)
                if (orow_own >= 0) {
                    const size_t o = (size_t)orow_own * p.ldc + n;
                    if (p.out_type == OUT_F16) {
                        __half2 h[16];
#pragma unroll
                        for (int i = 0; i < 16; ++i) h[i] = __floats2half2_rn(v[2 * i], v[2 * i + 1]);
                        uint4* dst = reinterpret_cast<uint4*>((__half*)p.C + o);
#pragma unroll
                        for (int i = 0; i < 4; ++i) if (8 * i < nv) dst[i] = *reinterpret_cast<uint4*>(&h[4 * i]);
                    } else {
                        __nv_bfloat162 h[16];
#pragma unroll
                        for (int i = 0; i < 16; ++i) h[i] = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
                        uint4* dst = reinterpret_cast<uint4*>((__nv_bfloat16*)p.C + o);
#pragma unroll
                        for (int i = 0; i < 4; ++i) if (8 * i < nv) dst[i] = *reinterpret_cast<uint4*>(&h[4 * i]);
                    }
                }
                continue;
            }
            __syncwarp();                                       // the previous chunk's reads of the patch are done
#pragma unroll
            for (int j = 0; j < 8; ++j) *reinterpret_cast<float4*>(stage + lane * EPI_RS + 4 * j) = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
            __syncwarp();
            if (c4 < nv) {
                float4 t[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) t[i] = *reinterpret_cast<const float4*>(stage + (4 * i + r4) * EPI_RS + c4);
                float* cbase = (p.epi == EPI_PARTIAL ? part_base : (float*)p.C) + n + c4;
                if (p.epi == EPI_RESID) {                       // x += alpha * t: all eight row loads in flight before the first store
                    float4 x[8];
#pragma unroll
                    for (int i = 0; i < 8; ++i) if (orow[i] >= 0) x[i] = *reinterpret_cast<const float4*>(cbase + (size_t)orow[i] * p.ldc);
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        if (orow[i] < 0) continue;
                        x[i].x += p.alpha * t[i].x; x[i].y += p.alpha * t[i].y; x[i].z += p.alpha * t[i].z; x[i].w += p.alpha * t[i].w;
                        *reinterpret_cast<float4*>(cbase + (size_t)orow[i] * p.ldc) = x[i];
                    }
                } else {
#pragma unroll
                    for (int i = 0; i < 8; ++i) if (orow[i] >= 0) *reinterpret_cast<float4*>(cbase + (size_t)orow[i] * p.ldc) = t[i];
                }
            }
        }
        if (tracer) trace_mark(trace_slot, 4);
}

template <int BN>
__device__ __forceinline__ void tc_epilogue(const TcParams& p, uint32_t tmem_base, uint64_t* tmem_full, int warp, int lane, int m0, int n0, int trace_slot,
                                            uint8_t* stage_base) {
    tc_epilogue_at<BN>(p, tmem_base, tmem_full, warp, m0 + (warp & 3) * 32, n0, trace_slot, stage_base);
}

template <int BN, int STAGES>
struct Smem {
    static_assert(STAGES * BM * ROW_BYTES >= EPI_STAGE_BYTES, "the epilogue patch lives in the A ring");
    alignas(1024) uint8_t a[STAGES][BM * ROW_BYTES];
    alignas(1024) uint8_t b[STAGES][BN * ROW_BYTES];
    alignas(8) uint64_t full[STAGES];
    uint64_t empty[STAGES];
    uint64_t tmem_full;
    uint32_t tmem_slot;
    int trace_slot;
};

// CL > 1: clusters of CL CTAs along N. Each CTA fetches 1/CL of every A tile and multicasts it to the whole cluster, so the
// activation tile crosses L2 -> SM once per cluster instead of once per CTA (at M = 128 the A re-reads, not the weights,
// dominate L2 traffic). A stage is refilled only when ALL CTAs of the cluster have consumed it: the MMA warp's commit
// arrives on the `empty` barrier of every CTA in the cluster (count CL).
template <int BN, int STAGES, int EB, int CL>
__global__ void __launch_bounds__(TC_THREADS, 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const TcParams p) {
    extern __shared__ uint8_t smem_raw[];
    using S = Smem<BN, STAGES>;
    S& s = *reinterpret_cast<S*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n0 = blockIdx.x * BN, m0 = blockIdx.y * BM;
    constexpr int BK = ROW_BYTES / EB;                                          // elements per k-block (64 for 16-bit, 32 for tf32)
    const int nk = p.K / BK / (int)gridDim.z;                                   // k-blocks of this split
    const int kb0 = (int)blockIdx.z * nk;
    const int rot = p.rot ? (int)((blockIdx.x / CL) % (unsigned)nk) : 0;  // k-block visited at loop index kb: kb0 + (kb + rot) % nk (same for a whole cluster)
    constexpr uint32_t TMEM_COLS = tmem_cols_for(BN);
    constexpr uint32_t STAGE_BYTES = (BM + BN) * ROW_BYTES;

    if (threadIdx.x == 0) {
        s.trace_slot = (blockIdx.x | blockIdx.y | blockIdx.z) == 0 ? trace_begin(TR_GEMM_TC) : -1;
        for (int i = 0; i < STAGES; ++i) { mbar_init(&s.full[i], 1); mbar_init(&s.empty[i], CL); }
        mbar_init(&s.tmem_full, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmA) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmB) : "memory");
    }
    if (warp == 2) tmem_alloc(&s.tmem_slot, TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    if (CL > 1) cluster_sync_all();                             // peers' barriers are initialised before any multicast / remote arrive
    tc_fence_after();
    const uint32_t tmem_base = s.tmem_slot;
    if (threadIdx.x == 0) { pdl_trigger(); trace_mark(s.trace_slot, 1); }   // the next kernel may start its own prologue / weight prefetch
    const uint32_t crank = CL > 1 ? cluster_ctarank() : 0;
    constexpr uint16_t MC_MASK = (uint16_t)((1u << CL) - 1);
    constexpr int A_SLICE_ROWS = BM / CL;
    auto load_a = [&](int st, int kc) {
        if (EB == 4 && p.a_fold) kc = kc < p.a_fold ? kc : kc - p.a_fold;
        if (CL > 1) tma_load_2d_mc(s.a[st] + crank * A_SLICE_ROWS * ROW_BYTES, &tmA, &s.full[st], kc, m0 + (int)crank * A_SLICE_ROWS, MC_MASK);
        else tma_load_2d(s.a[st], &tmA, &s.full[st], kc, m0);
    };

    if (warp == 0) {
        // ===================== TMA producer =====================
        if (elect_one()) {
            // Weights do not depend on the previous kernel: fill the ring with W tiles BEFORE waiting for it (PDL), so
            // HBM streaming of this GEMM overlaps the tail of its predecessor; A tiles follow after the wait.
            const int pre = nk < STAGES ? nk : STAGES;
            if (p.w_dyn) pdl_wait();
            for (int kb = 0; kb < pre; ++kb) {
                mbar_expect_tx(&s.full[kb], STAGE_BYTES);
                tma_load_2d(s.b[kb], &tmB, &s.full[kb], (kb0 + (kb + rot) % nk) * BK, n0);
            }
            if (!p.w_dyn) {
                for (int kb = pre; kb < nk; ++kb) tma_prefetch_2d(&tmB, (kb0 + (kb + rot) % nk) * BK, n0);   // rest of the slab: HBM -> L2 now
                pdl_wait();
            }
            for (int kb = 0; kb < pre; ++kb) load_a(kb, (kb0 + (kb + rot) % nk) * BK);
            for (int kb = pre; kb < nk; ++kb) {
                const int st = kb % STAGES; const uint32_t ph = (kb / STAGES) & 1;
                mbar_wait(&s.empty[st], ph ^ 1);
                mbar_expect_tx(&s.full[st], STAGE_BYTES);
                const int kc = (kb0 + (kb + rot) % nk) * BK;
                load_a(st, kc);
                tma_load_2d(s.b[st], &tmB, &s.full[st], kc, n0);
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer =====================
        if (elect_one()) {
            const uint32_t idesc = make_idesc(p.fmt, BN);
            for (int kb = 0; kb < nk; ++kb) {
                const int st = kb % STAGES; const uint32_t ph = (kb / STAGES) & 1;
                mbar_wait(&s.full[st], ph);
                tc_fence_after();
                const uint32_t a_addr = smem_u32(s.a[st]), b_addr = smem_u32(s.b[st]);
#pragma unroll
                for (int k = 0; k < ROW_BYTES / UMMA_K_BYTES; ++k) {
                    if (EB == 4) umma_tf32(tmem_base, make_desc(a_addr + k * UMMA_K_BYTES), make_desc(b_addr + k * UMMA_K_BYTES), idesc, (kb | k) ? 1u : 0u);
                    else umma_f16(tmem_base, make_desc(a_addr + k * UMMA_K_BYTES), make_desc(b_addr + k * UMMA_K_BYTES), idesc, (kb | k) ? 1u : 0u);
                }
                if (CL > 1) umma_commit_mc(&s.empty[st], MC_MASK);   // stage reusable cluster-wide once these MMAs retire
                else umma_commit(&s.empty[st]);                 // smem stage reusable once these MMAs retire
            }
            umma_commit(&s.tmem_full);                          // accumulator complete
        }
    } else {
        // ===================== epilogue =====================
        tc_epilogue<BN>(p, tmem_base, &s.tmem_full, warp, lane, m0, n0, s.trace_slot, s.a[0]);
    }
    tc_fence_before();
    __syncthreads();
    if (CL > 1) cluster_sync_all();                             // no CTA leaves while a peer's commit may still arrive on its barriers
    if (warp == 2) tmem_dealloc(tmem_base, TMEM_COLS);
}


// ------------------------------------------------------------------------------------------
// CTA-pair variant for small batches (one or few 128-row tiles): a cluster of two CTAs on neighbouring SMs computes one
// 128 x BN tile with tcgen05.mma.cta_group::2 (M = 128 across the pair). CTA r stages rows [64 r, 64 r + 64) of the activation
// tile and rows [r BN/2, (r+1) BN/2) of the weight tile; the tensor cores of both SMs read both halves of W, each SM
// accumulates its 64 rows. What this buys at M = 128: a CTA ingests HALF the activation tile (128 KB instead of 256 KB for
// K = 1024), and L2 -> SM ingest per SM is what bounds these GEMMs (DESIGN.md section 5).
//   * the `full` barriers live in CTA 0: both CTAs' TMA loads complete_tx there (cta_group::2 TMA, peer bit of the barrier
//     address cleared), CTA 0 arms them with the bytes of both halves and issues every MMA;
//   * tcgen05.commit.cta_group::2 ... multicast arrives on the `empty` / `tmem_full` barriers of BOTH CTAs;
//   * accumulator layout per CTA (cute tmem_frg_2sm, M_MMA = 64): lanes 0-63 = its 64 rows x columns [0, BN/2),
//     lanes 64-127 = the same rows x columns [BN/2, BN), BN/2 TMEM columns.
// ------------------------------------------------------------------------------------------
template <int BN, int STAGES>
struct SmemPair {
    static_assert(STAGES * 64 * ROW_BYTES >= EPI_STAGE_BYTES, "the epilogue patch lives in the A ring");
    alignas(1024) uint8_t a[STAGES][64 * ROW_BYTES];
    alignas(1024) uint8_t b[STAGES][(BN / 2) * ROW_BYTES];
    alignas(8) uint64_t full[STAGES];
    uint64_t empty[STAGES];
    uint64_t tmem_full;
    uint32_t tmem_slot;
    int trace_slot;
};

template <int BN, int STAGES>
__global__ void __launch_bounds__(TC_THREADS, 1)
gemm_tc_pair_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const TcParams p) {
    static_assert(BN % 64 == 0 && BN <= 256, "pair tile: BN/2 accumulator columns per lane half, read 32 at a time");
    extern __shared__ uint8_t smem_raw[];
    using S = SmemPair<BN, STAGES>;
    S& s = *reinterpret_cast<S*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = cluster_ctarank();                                    // 0 = leader (issues the MMAs, owns the full barriers)
    const int n0 = (int)(blockIdx.x >> 1) * BN, m0 = blockIdx.y * BM;
    constexpr int BK = ROW_BYTES / 2;                                           // 64 elements of 16 bits
    const int nk = p.K / BK / (int)gridDim.z;
    const int kb0 = (int)blockIdx.z * nk;
    constexpr uint32_t TMEM_COLS = BN / 2 < 32 ? 32 : BN / 2;
    constexpr uint32_t HALF_BYTES = (64 + BN / 2) * ROW_BYTES;                  // what ONE CTA stages per k-block

    if (threadIdx.x == 0) {
        s.trace_slot = (blockIdx.x | blockIdx.y | blockIdx.z) == 0 ? trace_begin(TR_GEMM_TC) : -1;
        for (int i = 0; i < STAGES; ++i) { mbar_init(&s.full[i], 1); mbar_init(&s.empty[i], 1); }
        mbar_init(&s.tmem_full, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmA) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmB) : "memory");
    }
    if (warp == 2) tmem_alloc_pair(&s.tmem_slot, TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();                                                         // both CTAs' barriers and TMEM are set up before any cross-CTA traffic
    tc_fence_after();
    const uint32_t tmem_base = s.tmem_slot;
    if (threadIdx.x == 0) { pdl_trigger(); trace_mark(s.trace_slot, 1); }

    if (warp == 0) {
        // ===================== TMA producer (both CTAs, each its halves) =====================
        if (elect_one()) {
            const int a_row = m0 + (int)rank * 64, b_row = n0 + (int)rank * (BN / 2);
            const int pre = nk < STAGES ? nk : STAGES;
            for (int kb = 0; kb < pre; ++kb) {                                  // weights first: they do not depend on the previous kernel
                if (rank == 0) mbar_expect_tx(&s.full[kb], 2 * HALF_BYTES);
                tma_load_2d_pair(s.b[kb], &tmB, &s.full[kb], (kb0 + kb) * BK, b_row);
            }
            for (int kb = pre; kb < nk; ++kb) tma_prefetch_2d(&tmB, (kb0 + kb) * BK, b_row);
            pdl_wait();
            for (int kb = 0; kb < pre; ++kb) tma_load_2d_pair(s.a[kb], &tmA, &s.full[kb], (kb0 + kb) * BK, a_row);
            for (int kb = pre; kb < nk; ++kb) {
                const int st = kb % STAGES; const uint32_t ph = (kb / STAGES) & 1;
                mbar_wait(&s.empty[st], ph ^ 1);                                // released for both CTAs by the leader's multicast commit
                if (rank == 0) mbar_expect_tx(&s.full[st], 2 * HALF_BYTES);
                tma_load_2d_pair(s.a[st], &tmA, &s.full[st], (kb0 + kb) * BK, a_row);
                tma_load_2d_pair(s.b[st], &tmB, &s.full[st], (kb0 + kb) * BK, b_row);
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer (leader CTA only) =====================
        if (rank == 0 && elect_one()) {
            const uint32_t idesc = make_idesc(p.fmt, BN);                       // M = 128 across the pair, N = BN
            for (int kb = 0; kb < nk; ++kb) {
                const int st = kb % STAGES; const uint32_t ph = (kb / STAGES) & 1;
                mbar_wait(&s.full[st], ph);                                     // both CTAs' halves of this k-block have landed
                tc_fence_after();
                const uint32_t a_addr = smem_u32(s.a[st]), b_addr = smem_u32(s.b[st]);
#pragma unroll
                for (int k = 0; k < ROW_BYTES / UMMA_K_BYTES; ++k)
                    umma_f16_pair(tmem_base, make_desc(a_addr + k * UMMA_K_BYTES), make_desc(b_addr + k * UMMA_K_BYTES), idesc, (kb | k) ? 1u : 0u);
                umma_commit_pair(&s.empty[st]);
            }
            umma_commit_pair(&s.tmem_full);
        }
    } else {
        // ===================== epilogue (both CTAs: 64 rows x BN columns each) =====================
        const int q = warp & 3;
        const int row0 = m0 + (int)rank * 64 + (q & 1) * 32;                    // TMEM lanes 32 q ..
        tc_epilogue_at<BN / 2>(p, tmem_base, &s.tmem_full, warp, row0, n0 + (q >> 1) * (BN / 2), s.trace_slot, s.a[0]);
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();                                                         // the peer's MMAs / commits may still touch this CTA's smem and barriers
    if (warp == 2) tmem_dealloc_pair(tmem_base, TMEM_COLS);
}

// ------------------------------------------------------------------------------------------
// CTA-pair variant for LARGE batches (>= ~4 row tiles; configs 3 and 5): a cluster of two CTAs computes one 256 x BN tile with
// tcgen05.mma.cta_group::2 at M = 256. CTA r stages rows [128 r, 128 r + 128) of the activation tile and rows
// [r BN/2, (r+1) BN/2) of the weight tile, and accumulates its 128 rows x BN columns (TMEM lane = row, as in the single-CTA tile).
// Why: at these batch sizes the single-CTA 128 x BN tile is bound by L2 -> SM ingest, not by the tensor pipe -- it pulls
// (128 + BN) x 128 B per k-block for 2 BN tensor-core clocks (96 B/clk at BN = 256, against ~60 B/clk that an SM sustains from L2:
// the 128 x 256 tile tops out near 64 % of the tensor peak). The pair tile pulls (128 + BN/2) x 128 B for the same 2 BN clocks
// per SM (64 B/clk at BN = 256). BN is any multiple of 16 (the epilogue masks the overhang of the last tile along N), chosen
// per shape so that the number of pair tiles lands just under a multiple of the 74 SM pairs (launch_gemm_tc). Stage counts keep
// the footprint <= ~107 KB: two CTAs of different pairs share an SM, one's epilogue hides behind the other's main loop.
// Barrier protocol = gemm_tc_pair_kernel's.
// ------------------------------------------------------------------------------------------
template <int BN, int STAGES>
struct SmemPair2 {
    alignas(1024) uint8_t a[STAGES][BM * ROW_BYTES];
    alignas(1024) uint8_t b[STAGES][(BN / 2) * ROW_BYTES];
    alignas(8) uint64_t full[STAGES];
    uint64_t empty[STAGES];
    uint64_t tmem_full;
    uint32_t tmem_slot;
    int trace_slot;
};

template <int BN, int STAGES>
__global__ void __launch_bounds__(TC_THREADS, 1)
gemm_tc_pair256_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const TcParams p) {
    static_assert(BN % 16 == 0 && BN >= 32 && BN <= 256, "pair256 tile: UMMA N is a multiple of 16 up to 256");
    extern __shared__ uint8_t smem_raw[];
    using S = SmemPair2<BN, STAGES>;
    S& s = *reinterpret_cast<S*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = cluster_ctarank();                                    // 0 = leader (issues the MMAs, owns the full barriers)
    const int n0 = (int)(blockIdx.x >> 1) * BN, m0 = blockIdx.y * (2 * BM);
    constexpr int BK = ROW_BYTES / 2;                                           // 64 elements of 16 bits
    const int nk = p.K / BK / (int)gridDim.z;
    const int kb0 = (int)blockIdx.z * nk;
    constexpr uint32_t TMEM_COLS = tmem_cols_for(BN);
    constexpr uint32_t HALF_BYTES = (BM + BN / 2) * ROW_BYTES;                  // what ONE CTA stages per k-block

    if (threadIdx.x == 0) {
        s.trace_slot = (blockIdx.x | blockIdx.y | blockIdx.z) == 0 ? trace_begin(TR_GEMM_TC) : -1;
        for (int i = 0; i < STAGES; ++i) { mbar_init(&s.full[i], 1); mbar_init(&s.empty[i], 1); }
        mbar_init(&s.tmem_full, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmA) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmB) : "memory");
    }
    if (warp == 2) tmem_alloc_pair(&s.tmem_slot, TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();                                                         // both CTAs' barriers and TMEM are set up before any cross-CTA traffic
    tc_fence_after();
    const uint32_t tmem_base = s.tmem_slot;
    if (threadIdx.x == 0) { pdl_trigger(); trace_mark(s.trace_slot, 1); }

    if (warp == 0) {
        // ===================== TMA producer (both CTAs, each its halves) =====================
        if (elect_one()) {
            const int a_row = m0 + (int)rank * BM, b_row = n0 + (int)rank * (BN / 2);
            const int pre = nk < STAGES ? nk : STAGES;
            if (p.w_dyn) pdl_wait();                                            // W written by the previous kernel (Q8_0 pre-dequantisation)
            for (int kb = 0; kb < pre; ++kb) {                                  // weights first: they do not depend on the previous kernel
                if (rank == 0) mbar_expect_tx(&s.full[kb], 2 * HALF_BYTES);
                tma_load_2d_pair(s.b[kb], &tmB, &s.full[kb], (kb0 + kb) * BK, b_row);
            }
            if (!p.w_dyn) pdl_wait();
            for (int kb = 0; kb < pre; ++kb) tma_load_2d_pair(s.a[kb], &tmA, &s.full[kb], (kb0 + kb) * BK, a_row);
            for (int kb = pre; kb < nk; ++kb) {
                const int st = kb % STAGES; const uint32_t ph = (kb / STAGES) & 1;
                mbar_wait(&s.empty[st], ph ^ 1);                                // released for both CTAs by the leader's multicast commit
                if (rank == 0) mbar_expect_tx(&s.full[st], 2 * HALF_BYTES);
                tma_load_2d_pair(s.a[st], &tmA, &s.full[st], (kb0 + kb) * BK, a_row);
                tma_load_2d_pair(s.b[st], &tmB, &s.full[st], (kb0 + kb) * BK, b_row);
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer (leader CTA only) =====================
        if (rank == 0 && elect_one()) {
            const uint32_t idesc = make_idesc(p.fmt, BN, 2 * BM);               // M = 256 across the pair, N = BN
            for (int kb = 0; kb < nk; ++kb) {
                const int st = kb % STAGES; const uint32_t ph = (kb / STAGES) & 1;
                mbar_wait(&s.full[st], ph);                                     // both CTAs' halves of this k-block have landed
                tc_fence_after();
                const uint32_t a_addr = smem_u32(s.a[st]), b_addr = smem_u32(s.b[st]);
#pragma unroll
                for (int k = 0; k < ROW_BYTES / UMMA_K_BYTES; ++k)
                    umma_f16_pair(tmem_base, make_desc(a_addr + k * UMMA_K_BYTES), make_desc(b_addr + k * UMMA_K_BYTES), idesc, (kb | k) ? 1u : 0u);
                umma_commit_pair(&s.empty[st]);
            }
            umma_commit_pair(&s.tmem_full);
        }
    } else {
        // ===================== epilogue (both CTAs: 128 rows x BN columns each) =====================
        tc_epilogue_at<BN>(p, tmem_base, &s.tmem_full, warp, m0 + (int)rank * BM + (warp & 3) * 32, n0, s.trace_slot, s.a[0]);
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();                                                         // the peer's MMAs / commits may still touch this CTA's smem and barriers
    if (warp == 2) tmem_dealloc_pair(tmem_base, TMEM_COLS);
}

// ------------------------------------------------------------------------------------------
// The same 256 x BN pair tile as a PERSISTENT kernel: one CTA pair per SM pair walks the (k-slice, m, n) tiles of the problem
// (n fastest: the pairs running side by side share the A rows in L2), with TWO accumulators in tensor memory (2 x up to 256 columns =
// all of it: one CTA per SM). The TMA ring never drains between tiles, the MMA warp starts tile i + 1 into the other accumulator as
// soon as its operands land, and the epilogue warps of both CTAs drain tile i meanwhile -- what the one-tile kernel above gets only
// from a second co-resident CTA (at half the shared memory = half the stages each). The epilogue patch has its own shared memory.
// Barriers: full / empty per stage as above; tmem_full[acc] (leader's commit, multicast to both CTAs) and tmem_empty[acc] in the
// LEADER (8 arrivals: the four epilogue warps of each CTA, the peer's through mapa + a cluster-scope arrive).
// ------------------------------------------------------------------------------------------
template <int BN, int STAGES>
struct SmemPairP {
    alignas(1024) uint8_t a[STAGES][BM * ROW_BYTES];
    alignas(1024) uint8_t b[STAGES][(BN / 2) * ROW_BYTES];
    alignas(16) uint8_t epi[EPI_STAGE_BYTES];
    alignas(8) uint64_t full[STAGES];
    uint64_t empty[STAGES];
    uint64_t tmem_full[2];
    uint64_t tmem_empty[2];
    uint32_t tmem_slot;
    int trace_slot;
};
__device__ __forceinline__ void mbar_arrive_cluster(uint64_t* bar, uint32_t cta) {    // arrive on the barrier at this offset in CTA `cta` of the cluster
    uint32_t remote;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(smem_u32(bar)), "r"(cta));
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(remote) : "memory");
}

template <int BN, int STAGES>
__global__ void __launch_bounds__(TC_THREADS, 1)
gemm_tc_pair256_persist_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const TcParams p, int tiles_n, int tiles_m,
                               int splits) {
    static_assert(BN % 16 == 0 && BN >= 32 && BN <= 256, "pair256 tile: UMMA N is a multiple of 16 up to 256");
    extern __shared__ uint8_t smem_raw[];
    using S = SmemPairP<BN, STAGES>;
    S& s = *reinterpret_cast<S*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = cluster_ctarank();
    const int pair = (int)(blockIdx.x >> 1), npairs = (int)(gridDim.x >> 1);
    constexpr int BK = ROW_BYTES / 2;
    const int nk = p.K / BK / splits;
    const int total = tiles_n * tiles_m * splits;
    constexpr uint32_t ACC_COLS = tmem_cols_for(BN);
    constexpr uint32_t HALF_BYTES = (BM + BN / 2) * ROW_BYTES;

    if (threadIdx.x == 0) {
        s.trace_slot = blockIdx.x == 0 ? trace_begin(TR_GEMM_TC) : -1;
        for (int i = 0; i < STAGES; ++i) { mbar_init(&s.full[i], 1); mbar_init(&s.empty[i], 1); }
        for (int i = 0; i < 2; ++i) { mbar_init(&s.tmem_full[i], 1); mbar_init(&s.tmem_empty[i], 8); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmA) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmB) : "memory");
    }
    if (warp == 2) tmem_alloc_pair(&s.tmem_slot, 2 * ACC_COLS);
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    tc_fence_after();
    const uint32_t tmem_base = s.tmem_slot;
    if (threadIdx.x == 0) { pdl_trigger(); trace_mark(s.trace_slot, 1); }
    // tile w -> k-slice z, m tile, n tile (n fastest)
    auto tile_of = [&](int w, int& z, int& m0, int& n0) {
        const int nt = w % tiles_n, r = w / tiles_n;
        z = r / tiles_m; m0 = (r % tiles_m) * (2 * BM); n0 = nt * BN;
    };

    if (warp == 0) {
        // ===================== TMA producer (both CTAs, each its halves): one ring across all tiles =====================
        if (elect_one()) {
            int g = 0;                                                          // k-blocks issued so far
            bool waited = false;
            for (int w = pair; w < total; w += npairs) {
                int z, m0, n0; tile_of(w, z, m0, n0);
                const int a_row = m0 + (int)rank * BM, b_row = n0 + (int)rank * (BN / 2), kb0 = z * nk;
                int kb = 0;
                if (!waited) {
                    // first tile: weights of the first stages BEFORE the dependency wait (they do not depend on the previous kernel)
                    const int pre = nk < STAGES ? nk : STAGES;
                    if (p.w_dyn) pdl_wait();
                    for (int i = 0; i < pre; ++i) {
                        if (rank == 0) mbar_expect_tx(&s.full[i], 2 * HALF_BYTES);
                        tma_load_2d_pair(s.b[i], &tmB, &s.full[i], (kb0 + i) * BK, b_row);
                    }
                    if (!p.w_dyn) pdl_wait();
                    for (int i = 0; i < pre; ++i) tma_load_2d_pair(s.a[i], &tmA, &s.full[i], (kb0 + i) * BK, a_row);
                    kb = pre; g = pre; waited = true;
                }
                for (; kb < nk; ++kb, ++g) {
                    const int st = g % STAGES; const uint32_t ph = (g / STAGES) & 1;
                    if (g >= STAGES) mbar_wait(&s.empty[st], ph ^ 1);
                    if (rank == 0) mbar_expect_tx(&s.full[st], 2 * HALF_BYTES);
                    tma_load_2d_pair(s.a[st], &tmA, &s.full[st], (kb0 + kb) * BK, a_row);
                    tma_load_2d_pair(s.b[st], &tmB, &s.full[st], (kb0 + kb) * BK, b_row);
                }
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer (leader CTA only) =====================
        if (rank == 0 && elect_one()) {
            const uint32_t idesc = make_idesc(p.fmt, BN, 2 * BM);
            int g = 0, it = 0;
            for (int w = pair; w < total; w += npairs, ++it) {
                const uint32_t acc = it & 1;
                mbar_wait(&s.tmem_empty[acc], (((uint32_t)it >> 1) & 1) ^ 1);   // both CTAs' epilogue warps have drained this accumulator (free at first use)
                tc_fence_after();
                const uint32_t tmem_c = tmem_base + acc * ACC_COLS;
                for (int kb = 0; kb < nk; ++kb, ++g) {
                    const int st = g % STAGES; const uint32_t ph = (g / STAGES) & 1;
                    mbar_wait(&s.full[st], ph);
                    tc_fence_after();
                    const uint32_t a_addr = smem_u32(s.a[st]), b_addr = smem_u32(s.b[st]);
#pragma unroll
                    for (int k = 0; k < ROW_BYTES / UMMA_K_BYTES; ++k)
                        umma_f16_pair(tmem_c, make_desc(a_addr + k * UMMA_K_BYTES), make_desc(b_addr + k * UMMA_K_BYTES), idesc, (kb | k) ? 1u : 0u);
                    umma_commit_pair(&s.empty[st]);
                }
                umma_commit_pair(&s.tmem_full[acc]);
            }
        }
    } else {
        // ===================== epilogue (both CTAs: 128 rows x BN columns of every tile) =====================
        int it = 0;
        for (int w = pair; w < total; w += npairs, ++it) {
            int z, m0, n0; tile_of(w, z, m0, n0);
            const uint32_t acc = it & 1;
            tc_epilogue_at<BN>(p, tmem_base + acc * ACC_COLS, &s.tmem_full[acc], warp, m0 + (int)rank * BM + (warp & 3) * 32, n0, it == 0 ? s.trace_slot : -1,
                               s.epi, ((uint32_t)it >> 1) & 1, z);
            tc_fence_before();                                                  // this warp's tcgen05.ld of the accumulator are complete (wait::ld inside)
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster(&s.tmem_empty[acc], 0);
        }
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    if (warp == 2) tmem_dealloc_pair(tmem_base, 2 * ACC_COLS);
}

// ------------------------------------------------------------------------------------------
// Q8_0 weights with the dequantisation fused into the operand path. The weight stays in HBM as the GGUF holds it, split
// into two planes at load (int8 quants [N][K], fp16 block scales [N][K/32]; the 34-byte blocks are not TMA-friendly).
// Per k-block: TMA brings the A tile (fp16, swizzled) and the RAW int8 W tile [BN][64]; warps 2-5 turn it into the fp16
// K-major SWIZZLE_128B tile the tensor core reads -- value = fp16(d) * q rounded to fp16, exactly what a load-time
// dequantisation to fp16 would hold -- fence it to the async proxy and signal the MMA warp. HBM traffic per weight is
// 1.0625 bytes instead of 2. The same warps run the epilogue afterwards.
// ------------------------------------------------------------------------------------------
template <int BN, int STAGES>
struct SmemQ8 {
    alignas(1024) uint8_t a[STAGES][BM * ROW_BYTES];
    alignas(1024) uint8_t b[STAGES][BN * ROW_BYTES];            // dequantised tile
    alignas(128) uint8_t q[STAGES][BN * 64];                    // raw quants, row-major [BN][64]
    alignas(16) __half sc[BN * 128];                            // block scales of this CTA's k range: [BN][2 * nk], nk <= 64
    alignas(8) uint64_t full[STAGES];
    uint64_t bready[STAGES];
    uint64_t empty[STAGES];
    uint64_t tmem_full;
    uint32_t tmem_slot;
    int trace_slot;
};

// Q4 = 1: the same pipeline for Q4_0 weights (scripts/convert_to_gguf.py:132-179): the raw tile is [BN][32] bytes of nibbles per
// k-block (two 32-value blocks; byte i of a block = value i in the low nibble, value i + 16 in the high one, stored value q in 0..15
// meaning q - 8), the dequantiser expands fp16(d) * (q - 8) -- HBM traffic per weight 0.5625 bytes.
template <int BN, int STAGES, int Q4>
__global__ void __launch_bounds__(Q8_THREADS, 1)
gemm_q8_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmQ, const __half* __restrict__ scales,
               const TcParams p) {
    extern __shared__ uint8_t smem_raw[];
    using S = SmemQ8<BN, STAGES>;
    S& s = *reinterpret_cast<S*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n0 = blockIdx.x * BN, m0 = blockIdx.y * BM;
    constexpr int BK = 64;
    const int nk = p.K / BK / (int)gridDim.z;
    const int kb0 = (int)blockIdx.z * nk;
    const int rot = p.rot ? (int)(blockIdx.x % (unsigned)nk) : 0;
    constexpr uint32_t TMEM_COLS = BN < 32 ? 32 : BN;
    constexpr int QROW = Q4 ? 32 : 64;                                          // raw bytes per weight row and k-block
    constexpr uint32_t STAGE_BYTES = BM * ROW_BYTES + BN * QROW;

    if (threadIdx.x == 0) {
        s.trace_slot = (blockIdx.x | blockIdx.y | blockIdx.z) == 0 ? trace_begin(TR_GEMM_Q8) : -1;
        for (int i = 0; i < STAGES; ++i) { mbar_init(&s.full[i], 1); mbar_init(&s.bready[i], Q8_DEQ); mbar_init(&s.empty[i], 1); }
        mbar_init(&s.tmem_full, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmA) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmQ) : "memory");
    }
    if (warp == 2) tmem_alloc(&s.tmem_slot, TMEM_COLS);
    if (warp >= 2) {                                             // block scales of this tile's k range (static data: before the PDL wait)
        const int t = threadIdx.x - 64, per_row = 2 * nk;
        const __half* src0 = scales + (size_t)n0 * (p.K / 32) + (size_t)kb0 * 2;
        if ((nk & 1) == 0) {                                     // 8-byte vectors: one round trip for the whole tile
            const int vpr = per_row / 4;
            for (int e = t; e < BN * vpr; e += Q8_DEQ) {
                const int r = e / vpr, j = e % vpr;
                *reinterpret_cast<uint2*>(&s.sc[r * per_row + j * 4]) = __ldg(reinterpret_cast<const uint2*>(src0 + (size_t)r * (p.K / 32) + j * 4));
            }
        } else {
            for (int e = t; e < BN * per_row; e += Q8_DEQ) {
                const int r = e / per_row, j = e % per_row;
                s.sc[r * per_row + j] = src0[(size_t)r * (p.K / 32) + j];
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = s.tmem_slot;
    if (threadIdx.x == 0) { pdl_trigger(); trace_mark(s.trace_slot, 1); }

    if (warp == 0) {
        // ===================== TMA producer =====================
        if (elect_one()) {
            const int pre = nk < STAGES ? nk : STAGES;
            for (int kb = 0; kb < pre; ++kb) {
                mbar_expect_tx(&s.full[kb], STAGE_BYTES);
                tma_load_2d(s.q[kb], &tmQ, &s.full[kb], (kb0 + (kb + rot) % nk) * QROW, n0);
            }
            for (int kb = pre; kb < nk; ++kb) tma_prefetch_2d(&tmQ, (kb0 + (kb + rot) % nk) * QROW, n0);
            pdl_wait();
            for (int kb = 0; kb < pre; ++kb) tma_load_2d(s.a[kb], &tmA, &s.full[kb], (kb0 + (kb + rot) % nk) * BK, m0);
            for (int kb = pre; kb < nk; ++kb) {
                const int st = kb % STAGES; const uint32_t ph = (kb / STAGES) & 1;
                mbar_wait(&s.empty[st], ph ^ 1);
                mbar_expect_tx(&s.full[st], STAGE_BYTES);
                const int kc = (kb0 + (kb + rot) % nk) * BK;
                tma_load_2d(s.a[st], &tmA, &s.full[st], kc, m0);
                tma_load_2d(s.q[st], &tmQ, &s.full[st], kc / BK * QROW, n0);
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer =====================
        if (elect_one()) {
            const uint32_t idesc = make_idesc(0, BN);
            for (int kb = 0; kb < nk; ++kb) {
                const int st = kb % STAGES; const uint32_t ph = (kb / STAGES) & 1;
                mbar_wait(&s.full[st], ph);                     // A tile landed
                mbar_wait(&s.bready[st], ph);                   // W tile dequantised
                tc_fence_after();
                const uint32_t a_addr = smem_u32(s.a[st]), b_addr = smem_u32(s.b[st]);
#pragma unroll
                for (int k = 0; k < ROW_BYTES / UMMA_K_BYTES; ++k)
                    umma_f16(tmem_base, make_desc(a_addr + k * UMMA_K_BYTES), make_desc(b_addr + k * UMMA_K_BYTES), idesc, (kb | k) ? 1u : 0u);
                umma_commit(&s.empty[st]);
            }
            umma_commit(&s.tmem_full);
        }
    } else {
        // ===================== dequantiser (then epilogue) =====================
        const int t = threadIdx.x - 64;                          // 0..255: 64 rows x 4 sixteen-byte chunks per pass
        const int c = t & 3, per_row = 2 * nk;
        for (int kb = 0; kb < nk; ++kb) {
            const int st = kb % STAGES; const uint32_t ph = (kb / STAGES) & 1;
            const int kk = (kb + rot) % nk;                     // k-block of this stage within the CTA's range
            mbar_wait(&s.full[st], ph);
#pragma unroll
            for (int pz = 0; pz < (BN + 63) / 64; ++pz) {
                const int r = pz * 64 + (t >> 2);
                if (BN % 64 != 0 && r >= BN) continue;                             // BN = 32: only the first 128 threads have a row
                // 16 weights per thread: Q8_0 = 16 bytes of the row; Q4_0 = the 16 low (c even) or high (c odd) nibbles of block c / 2
                uint4 raw = *reinterpret_cast<const uint4*>(&s.q[st][r * QROW + (Q4 ? (c >> 1) * 16 : c * 16)]);
                const __half2 d2 = __half2half2(s.sc[r * per_row + kk * 2 + (c >> 1)]);
                // int8 -> fp16 without integer conversions: q + 128 as the low mantissa bits of 1024.0 (0x6400 | byte), minus 1152;
                // then ONE fp16 multiply by the block scale = fp16(d) * q rounded once, exactly the value a load-time dequantisation
                // to fp16 holds. 7 instructions per 4 weights (the conversion path was what bound this kernel).
                if (Q4) {                                                             // nibble n -> byte n: then (0x6400 | n) - 1032 = n - 8
                    const int sh = (c & 1) * 4;
                    raw.x = (raw.x >> sh) & 0x0F0F0F0Fu; raw.y = (raw.y >> sh) & 0x0F0F0F0Fu; raw.z = (raw.z >> sh) & 0x0F0F0F0Fu; raw.w = (raw.w >> sh) & 0x0F0F0F0Fu;
                }
                const uint32_t w4[4] = {raw.x, raw.y, raw.z, raw.w};
                const __half2 off = Q4 ? __floats2half2_rn(1032.0f, 1032.0f) : __floats2half2_rn(1152.0f, 1152.0f);
                __half2 h[8];
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const uint32_t x = Q4 ? w4[i] : (w4[i] ^ 0x80808080u);
                    const uint32_t lo = __byte_perm(x, 0x64646464u, 0x5140), hi = __byte_perm(x, 0x64646464u, 0x5342);
                    h[2 * i] = __hmul2(__hsub2(*reinterpret_cast<const __half2*>(&lo), off), d2);
                    h[2 * i + 1] = __hmul2(__hsub2(*reinterpret_cast<const __half2*>(&hi), off), d2);
                }
                uint8_t* row = &s.b[st][r * ROW_BYTES];
                *reinterpret_cast<uint4*>(row + (((2 * c) ^ (r & 7)) << 4)) = *reinterpret_cast<uint4*>(&h[0]);      // SWIZZLE_128B: chunk ^= row % 8
                *reinterpret_cast<uint4*>(row + (((2 * c + 1) ^ (r & 7)) << 4)) = *reinterpret_cast<uint4*>(&h[4]);
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");          // generic-proxy writes -> visible to the tensor core
            asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(&s.bready[st])) : "memory");
        }
        if (warp < 6) tc_epilogue<BN>(p, tmem_base, &s.tmem_full, warp, lane, m0, n0, s.trace_slot, s.a[0]);
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 2) tmem_dealloc(tmem_base, TMEM_COLS);
}

// ------------------------------------------------------------------------------------------
// Q8_0 / Q4_0 weights on the 256-row CTA-pair tiles (large batches): the fused-dequantisation pipeline of gemm_q8_kernel inside the
// cta_group::2 structure of gemm_tc_pair256_kernel. Each CTA of the pair stages its 128 rows of A (fp16, TMA, counted on the leader's
// `full` barrier) and the RAW quants of its BN/2 weight rows (TMA into its own shared memory, its own `qfull` barrier); its four
// dequantiser warps expand them into the fp16 SWIZZLE_128B half-tile the pair's MMA reads and arrive on the CTA's own `bready` barrier;
// the peer CTA's (otherwise idle) MMA warp relays its barrier to the leader's `peer_ready` through mapa + a cluster-scope arrive. The same
// four warps run the epilogue afterwards. A weight is dequantised once per 256 output rows (the single-CTA
// kernel: once per 128) and crosses L2 -> SM as 1.06 (0.56) bytes instead of 2: on tiles whose main loop is bound by what an SM can
// ingest, the quantised operand is the FASTER one. Block scales are read straight from global memory one k-block ahead (4 bytes per
// row and k-block: no shared-memory table). Values = fp16(d) * q rounded once: identical to the other Q8_0 paths.
// ------------------------------------------------------------------------------------------
template <int BN, int STAGES, int Q4>
struct SmemQ8Pair {
    static constexpr int QROW = Q4 ? 32 : 64;
    alignas(1024) uint8_t a[STAGES][BM * ROW_BYTES];
    alignas(1024) uint8_t b[STAGES][(BN / 2) * ROW_BYTES];      // dequantised half tile
    alignas(128) uint8_t q[STAGES][(BN / 2) * QROW];            // raw quants of this CTA's weight rows
    alignas(8) uint64_t full[STAGES];                            // leader: both CTAs' A halves landed
    uint64_t qfull[STAGES];                                      // own: raw quants landed
    uint64_t bready[STAGES];                                     // own: this CTA's half tile dequantised (4 warp arrivals)
    uint64_t peer_ready[STAGES];                                 // leader: the peer's half tile dequantised (relayed by the peer's idle MMA warp)
    uint64_t empty[STAGES];
    uint64_t tmem_full;
    uint32_t tmem_slot;
    int trace_slot;
};

template <int BN, int STAGES, int Q4>
__global__ void __launch_bounds__(QP_THREADS, 2)
gemm_q8_pair256_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmQ, const __half* __restrict__ scales,
                       const TcParams p) {
    static_assert(BN % 16 == 0 && BN >= 32 && BN <= 256, "pair256 tile: UMMA N is a multiple of 16 up to 256");
    extern __shared__ uint8_t smem_raw[];
    using S = SmemQ8Pair<BN, STAGES, Q4>;
    S& s = *reinterpret_cast<S*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = cluster_ctarank();
    const int n0 = (int)(blockIdx.x >> 1) * BN, m0 = blockIdx.y * (2 * BM);
    constexpr int BK = 64, QROW = S::QROW, HB = BN / 2;
    const int nk = p.K / BK / (int)gridDim.z;
    const int kb0 = (int)blockIdx.z * nk;
    constexpr uint32_t TMEM_COLS = tmem_cols_for(BN);
    const int b_row = n0 + (int)rank * HB;                                       // this CTA's weight rows

    if (threadIdx.x == 0) {
        s.trace_slot = (blockIdx.x | blockIdx.y | blockIdx.z) == 0 ? trace_begin(TR_GEMM_Q8) : -1;
        for (int i = 0; i < STAGES; ++i) { mbar_init(&s.full[i], 1); mbar_init(&s.qfull[i], 1); mbar_init(&s.bready[i], QP_DEQ / 32); mbar_init(&s.peer_ready[i], 1); mbar_init(&s.empty[i], 1); }
        mbar_init(&s.tmem_full, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmA) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmQ) : "memory");
    }
    if (warp == 2) tmem_alloc_pair(&s.tmem_slot, TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    tc_fence_after();
    const uint32_t tmem_base = s.tmem_slot;
    if (threadIdx.x == 0) { pdl_trigger(); trace_mark(s.trace_slot, 1); }

    if (warp == 0) {
        // ===================== TMA producer (both CTAs) =====================
        if (elect_one()) {
            const int a_row = m0 + (int)rank * BM;
            const int pre = nk < STAGES ? nk : STAGES;
            for (int kb = 0; kb < pre; ++kb) {                                  // weights first: they do not depend on the previous kernel
                mbar_expect_tx(&s.qfull[kb], HB * QROW);
                tma_load_2d(s.q[kb], &tmQ, &s.qfull[kb], (kb0 + kb) * QROW, b_row);
                if (rank == 0) mbar_expect_tx(&s.full[kb], 2 * BM * ROW_BYTES);
            }
            pdl_wait();
            for (int kb = 0; kb < pre; ++kb) tma_load_2d_pair(s.a[kb], &tmA, &s.full[kb], (kb0 + kb) * BK, a_row);
            for (int kb = pre; kb < nk; ++kb) {
                const int st = kb % STAGES; const uint32_t ph = (kb / STAGES) & 1;
                mbar_wait(&s.empty[st], ph ^ 1);                                // the pair's MMAs on this stage have retired (multicast commit)
                mbar_expect_tx(&s.qfull[st], HB * QROW);
                tma_load_2d(s.q[st], &tmQ, &s.qfull[st], (kb0 + kb) * QROW, b_row);
                if (rank == 0) mbar_expect_tx(&s.full[st], 2 * BM * ROW_BYTES);
                tma_load_2d_pair(s.a[st], &tmA, &s.full[st], (kb0 + kb) * BK, a_row);
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer (leader CTA); in the peer CTA this warp relays "half tile dequantised" to the leader =====================
        if (rank != 0) {
            // one thread, nothing of its own in flight: the cluster-scope release of the remote arrive (a MEMBAR.GPU) costs it nothing, whereas
            // issued by the dequantiser warps themselves it was 20 % of the kernel's stall samples (and waited for their scale loads)
            if (elect_one()) {
                for (int kb = 0; kb < nk; ++kb) {
                    const int st = kb % STAGES; const uint32_t ph = (kb / STAGES) & 1;
                    mbar_wait(&s.bready[st], ph);                               // acquire: the dequantisers' (proxy-fenced) shared-memory writes are performed
                    // relaxed: nothing of THIS thread needs publishing, and the release form costs a MEMBAR.GPU round trip per k-block on the
                    // critical path of every stage (7.7 % of the kernel's stall samples, all of them here)
                    uint32_t remote;
                    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(smem_u32(&s.peer_ready[st])), "r"(0));
                    asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(remote) : "memory");
                }
            }
        } else if (elect_one()) {
            const uint32_t idesc = make_idesc(0, BN, 2 * BM);
            for (int kb = 0; kb < nk; ++kb) {
                const int st = kb % STAGES; const uint32_t ph = (kb / STAGES) & 1;
                mbar_wait(&s.full[st], ph);                                     // both A halves landed
                mbar_wait(&s.bready[st], ph);                                   // this CTA's W half tile dequantised
                mbar_wait(&s.peer_ready[st], ph);                               // the peer's
                tc_fence_after();
                const uint32_t a_addr = smem_u32(s.a[st]), b_addr = smem_u32(s.b[st]);
#pragma unroll
                for (int k = 0; k < ROW_BYTES / UMMA_K_BYTES; ++k)
                    umma_f16_pair(tmem_base, make_desc(a_addr + k * UMMA_K_BYTES), make_desc(b_addr + k * UMMA_K_BYTES), idesc, (kb | k) ? 1u : 0u);
                umma_commit_pair(&s.empty[st]);
            }
            umma_commit_pair(&s.tmem_full);
        }
    } else {
        // ===================== dequantiser (then epilogue) =====================
        const int t = threadIdx.x - 64;                                          // 0..127: 32 rows x 4 sixteen-value chunks per pass
        const int c = t & 3;
        constexpr int RPP = QP_DEQ / 4, PASSES = (HB + RPP - 1) / RPP;
        const int kblocks = p.K / 32;                                            // block scales per weight row
        // block scale of (row of pass pz, k-block kb): one half per thread, fetched one k-block ahead
        auto load_scale = [&](int pz, int kb) {
            const int r = pz * RPP + (t >> 2), n = b_row + r;
            return (r < HB && n < p.N) ? scales[(size_t)n * kblocks + (size_t)(kb0 + kb) * 2 + (c >> 1)] : __float2half(0.f);
        };
        __half d_cur[PASSES];                                                     // scales of the k-block about to be expanded: loaded right AFTER the previous
#pragma unroll                                                                   // k-block's arrive, so that no load is in flight at its fence, and consumed after the next barrier wait
        for (int pz = 0; pz < PASSES; ++pz) d_cur[pz] = load_scale(pz, 0);
        for (int kb = 0; kb < nk; ++kb) {
            const int st = kb % STAGES; const uint32_t ph = (kb / STAGES) & 1;
            mbar_wait(&s.qfull[st], ph);
#pragma unroll
            for (int pz = 0; pz < PASSES; ++pz) {
                const int r = pz * RPP + (t >> 2);
                if (HB % RPP != 0 && r >= HB) continue;
                uint4 raw = *reinterpret_cast<const uint4*>(&s.q[st][r * QROW + (Q4 ? (c >> 1) * 16 : c * 16)]);
                const __half2 d2 = __half2half2(d_cur[pz]);
                if (Q4) {
                    const int sh = (c & 1) * 4;
                    raw.x = (raw.x >> sh) & 0x0F0F0F0Fu; raw.y = (raw.y >> sh) & 0x0F0F0F0Fu; raw.z = (raw.z >> sh) & 0x0F0F0F0Fu; raw.w = (raw.w >> sh) & 0x0F0F0F0Fu;
                }
                const uint32_t w4[4] = {raw.x, raw.y, raw.z, raw.w};
                const __half2 off = Q4 ? __floats2half2_rn(1032.0f, 1032.0f) : __floats2half2_rn(1152.0f, 1152.0f);
                __half2 h[8];
#pragma unroll
                for (int i = 0; i < 4; ++i) {                                    // (0x6400 | byte) - offset = q exactly; one fp16 multiply by the block scale
                    const uint32_t x = Q4 ? w4[i] : (w4[i] ^ 0x80808080u);
                    const uint32_t lo = __byte_perm(x, 0x64646464u, 0x5140), hi = __byte_perm(x, 0x64646464u, 0x5342);
                    h[2 * i] = __hmul2(__hsub2(*reinterpret_cast<const __half2*>(&lo), off), d2);
                    h[2 * i + 1] = __hmul2(__hsub2(*reinterpret_cast<const __half2*>(&hi), off), d2);
                }
                uint8_t* row = &s.b[st][r * ROW_BYTES];
                *reinterpret_cast<uint4*>(row + (((2 * c) ^ (r & 7)) << 4)) = *reinterpret_cast<uint4*>(&h[0]);      // SWIZZLE_128B: chunk ^= row % 8
                *reinterpret_cast<uint4*>(row + (((2 * c + 1) ^ (r & 7)) << 4)) = *reinterpret_cast<uint4*>(&h[4]);
            }
            // generic-proxy writes -> visible to the tensor cores of the pair. The shared::cta form only: the unqualified fence also waits
            // for the scale load in flight for the next k-block (an L2 round trip per k-block: measured 2x the whole kernel)
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            __syncwarp();
            if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(&s.bready[st])) : "memory");
            if (kb + 1 < nk) {
#pragma unroll
                for (int pz = 0; pz < PASSES; ++pz) d_cur[pz] = load_scale(pz, kb + 1);
            }
        }
        tc_epilogue_at<BN>(p, tmem_base, &s.tmem_full, warp, m0 + (int)rank * BM + (warp & 3) * 32, n0, s.trace_slot, s.a[0]);
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    if (warp == 2) tmem_dealloc_pair(tmem_base, TMEM_COLS);
}

// ------------------------------------------------------------------ host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn get_encode_fn() {
    static EncodeTiledFn fn = nullptr;
    static std::once_flag once;
    std::call_once(once, [] {
        void* p = nullptr; cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess || !p)
            throw CudaError("cuTensorMapEncodeTiled entry point not available");
        fn = (EncodeTiledFn)p;
    });
    return fn;
}
// 2-D K-major tensor map: dims {K, rows}, row stride ld elements, box {64, box_rows}, 128-byte swizzle
CUtensorMap make_map(const void* ptr, int rows, int K, long long ld, int box_rows, int fmt) {
    CUtensorMap m;
    const int eb = fmt == 2 ? 4 : 2;
    const cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)rows};
    const cuuint64_t strides[1] = {(cuuint64_t)ld * eb};
    const cuuint32_t box[2] = {(cuuint32_t)(ROW_BYTES / eb), (cuuint32_t)box_rows};
    const cuuint32_t estr[2] = {1, 1};
    const CUtensorMapDataType dt = fmt == 2 ? CU_TENSOR_MAP_DATA_TYPE_TFLOAT32 : fmt == 1 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
    const CUresult r = get_encode_fn()(&m, dt, 2, const_cast<void*>(ptr),
                                       dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                                       CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) throw CudaError("cuTensorMapEncodeTiled failed (" + std::to_string((int)r) + ")");
    return m;
}

CUtensorMap make_map_u8(const void* ptr, int rows, int K, int box_rows, int box_cols = 64) {
    CUtensorMap m;
    const cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)rows};
    const cuuint64_t strides[1] = {(cuuint64_t)K};
    const cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
    const cuuint32_t estr[2] = {1, 1};
    const CUresult r = get_encode_fn()(&m, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                                       CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                                       CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) throw CudaError("cuTensorMapEncodeTiled (u8) failed (" + std::to_string((int)r) + ")");
    return m;
}

// the single-CTA and 128-row pair tiles launch N / BN column tiles: with N % BN != 0 the last columns would never be written
void require_full_grid(int N, int BN) {
    if (N % BN != 0) throw std::invalid_argument("gemm_tc: N = " + std::to_string(N) + " is not a multiple of the tile width " + std::to_string(BN));
}

template <int BN, int STAGES, int Q4>
void launch_cfg_q8x(const GemmArgs& a, cudaStream_t st) {
    static std::atomic<size_t> attr_set[MAX_DEVICES];
    const size_t smem = sizeof(SmemQ8<BN, STAGES>) + 1024;
    ensure_dyn_smem(gemm_q8_kernel<BN, STAGES, Q4>, smem, attr_set);
    if (a.K / 64 / a.splits > 64) throw CudaError("gemm_q8: k range per CTA too long for the scale buffer");
    const CUtensorMap tmA = make_map(a.A, a.M, a.K, a.lda, BM, 0);
    const CUtensorMap tmQ = Q4 ? make_map_u8(a.W, a.N, a.K / 2, BN, 32) : make_map_u8(a.W, a.N, a.K, BN);
    require_full_grid(a.N, BN);
    const int m_out = a.c_group > 0 ? (a.M / a.c_group) * (a.c_group - a.c_drop) : a.M;
    TcParams p{a.M, a.N, a.K, a.bias, a.C, a.ldc, a.epi, a.alpha, a.out_type, 0, a.rotate, a.c_group, a.c_drop, a.C0, m_out};
    dim3 grid(a.N / BN, (a.M + BM - 1) / BM, a.splits);
    launch_k(gemm_q8_kernel<BN, STAGES, Q4>, grid, dim3(Q8_THREADS), smem, st, tmA, tmQ, (const __half*)a.w_scales, p);
}
template <int BN, int STAGES>
void launch_cfg_q8(const GemmArgs& a, cudaStream_t st) { if (a.q4) launch_cfg_q8x<BN, STAGES, 1>(a, st); else launch_cfg_q8x<BN, STAGES, 0>(a, st); }

template <int BN, int STAGES, int Q4>
void launch_cfg_q8_pair256x(const GemmArgs& a, cudaStream_t st) {
    static std::atomic<size_t> attr_set[MAX_DEVICES];
    const size_t smem = sizeof(SmemQ8Pair<BN, STAGES, Q4>) + 1024;
    ensure_dyn_smem(gemm_q8_pair256_kernel<BN, STAGES, Q4>, smem, attr_set);
    const CUtensorMap tmA = make_map(a.A, a.M, a.K, a.lda, BM, 0);
    const CUtensorMap tmQ = Q4 ? make_map_u8(a.W, a.N, a.K / 2, BN / 2, 32) : make_map_u8(a.W, a.N, a.K, BN / 2, 64);
    const int m_out = a.c_group > 0 ? (a.M / a.c_group) * (a.c_group - a.c_drop) : a.M;
    TcParams p{a.M, a.N, a.K, a.bias, a.C, a.ldc, a.epi, a.alpha, a.out_type, 0, 0, a.c_group, a.c_drop, a.C0, m_out};
    dim3 grid(2 * ((a.N + BN - 1) / BN), (a.M + 2 * BM - 1) / (2 * BM), a.splits > 1 ? a.splits : 1);
    launch_k_cluster(gemm_q8_pair256_kernel<BN, STAGES, Q4>, grid, dim3(QP_THREADS), smem, st, 2, tmA, tmQ, (const __half*)a.w_scales, p);
}
void launch_q8_pair256(const GemmArgs& a, int bn, cudaStream_t st) {
    // stage counts: <= ~111 KB per CTA so that two CTAs of different pairs share an SM (16 KB A + BN/2 x (128 + 64) bytes per stage)
    switch (bn) {
        case 208: if (a.q4) launch_cfg_q8_pair256x<208, 3, 1>(a, st); else launch_cfg_q8_pair256x<208, 3, 0>(a, st); break;
        case 160: if (a.q4) launch_cfg_q8_pair256x<160, 3, 1>(a, st); else launch_cfg_q8_pair256x<160, 3, 0>(a, st); break;
        case 112: if (a.q4) launch_cfg_q8_pair256x<112, 4, 1>(a, st); else launch_cfg_q8_pair256x<112, 4, 0>(a, st); break;
        default: throw CudaError("gemm_q8: pair256 tile not instantiated");
    }
}
// Experimental, off by default: on B200 the multicast variant measured SLOWER than per-CTA A loads at M = 128
// (ff1a 7.7 vs 6.9 us, profiles/r01_notes.md) -- L2 already serves the shared tile well and the cluster-wide stage release
// couples the CTAs -- and it is not covered by the parity suite.
bool multicast_enabled() {
    static const bool on = [] { const char* e = getenv("NSB_MC"); return e && e[0] == '1'; }();
    return on;
}

template <int BN, int STAGES, int EB, int CL>
void launch_cfg_c(const GemmArgs& a, int fmt, cudaStream_t st) {
    static std::atomic<size_t> attr_set[MAX_DEVICES];
    require_full_grid(a.N, BN);
    const size_t smem = sizeof(Smem<BN, STAGES>) + 1024;
    ensure_dyn_smem(gemm_tc_kernel<BN, STAGES, EB, CL>, smem, attr_set);
    const CUtensorMap tmA = make_map(a.A, a.M, a.a_fold ? 2 * a.a_fold : a.K, a.lda, BM / CL, fmt);
    const CUtensorMap tmB = make_map(a.W, a.N, a.K, a.K, BN, fmt);
    const int m_out = a.c_group > 0 ? (a.M / a.c_group) * (a.c_group - a.c_drop) : a.M;
    TcParams p{a.M, a.N, a.K, a.bias, a.C, a.ldc, a.epi, a.alpha, a.out_type, fmt, a.rotate, a.c_group, a.c_drop, a.C0, m_out, a.w_dynamic, a.a_fold};
    dim3 grid(a.N / BN, (a.M + BM - 1) / BM, a.splits);
    launch_k_cluster(gemm_tc_kernel<BN, STAGES, EB, CL>, grid, dim3(TC_THREADS), smem, st, CL, tmA, tmB, p);
}
template <int BN, int STAGES>
void launch_cfg_pair(const GemmArgs& a, int fmt, cudaStream_t st) {
    static std::atomic<size_t> attr_set[MAX_DEVICES];
    require_full_grid(a.N, BN);
    const size_t smem = sizeof(SmemPair<BN, STAGES>) + 1024;
    ensure_dyn_smem(gemm_tc_pair_kernel<BN, STAGES>, smem, attr_set);
    const CUtensorMap tmA = make_map(a.A, a.M, a.K, a.lda, 64, fmt);
    const CUtensorMap tmB = make_map(a.W, a.N, a.K, a.K, BN / 2, fmt);
    const int m_out = a.c_group > 0 ? (a.M / a.c_group) * (a.c_group - a.c_drop) : a.M;
    TcParams p{a.M, a.N, a.K, a.bias, a.C, a.ldc, a.epi, a.alpha, a.out_type, fmt, 0, a.c_group, a.c_drop, a.C0, m_out};
    dim3 grid(2 * (a.N / BN), (a.M + BM - 1) / BM, a.splits);
    launch_k_cluster(gemm_tc_pair_kernel<BN, STAGES>, grid, dim3(TC_THREADS), smem, st, 2, tmA, tmB, p);
}

template <int BN, int STAGES>
void launch_cfg_pair256(const GemmArgs& a, int fmt, cudaStream_t st) {
    static std::atomic<size_t> attr_set[MAX_DEVICES];
    const size_t smem = sizeof(SmemPair2<BN, STAGES>) + 1024;
    ensure_dyn_smem(gemm_tc_pair256_kernel<BN, STAGES>, smem, attr_set);
    const CUtensorMap tmA = make_map(a.A, a.M, a.K, a.lda, BM, fmt);
    const CUtensorMap tmB = make_map(a.W, a.N, a.K, a.K, BN / 2, fmt);
    const int m_out = a.c_group > 0 ? (a.M / a.c_group) * (a.c_group - a.c_drop) : a.M;
    TcParams p{a.M, a.N, a.K, a.bias, a.C, a.ldc, a.epi, a.alpha, a.out_type, fmt, 0, a.c_group, a.c_drop, a.C0, m_out, a.w_dynamic};
    dim3 grid(2 * ((a.N + BN - 1) / BN), (a.M + 2 * BM - 1) / (2 * BM), a.splits);
    launch_k_cluster(gemm_tc_pair256_kernel<BN, STAGES>, grid, dim3(TC_THREADS), smem, st, 2, tmA, tmB, p);
}
template <int BN, int STAGES>
void launch_cfg_pair256_persist(const GemmArgs& a, int fmt, cudaStream_t st) {
    static std::atomic<size_t> attr_set[MAX_DEVICES];
    const size_t smem = sizeof(SmemPairP<BN, STAGES>) + 1024;
    ensure_dyn_smem(gemm_tc_pair256_persist_kernel<BN, STAGES>, smem, attr_set);
    const CUtensorMap tmA = make_map(a.A, a.M, a.K, a.lda, BM, fmt);
    const CUtensorMap tmB = make_map(a.W, a.N, a.K, a.K, BN / 2, fmt);
    const int m_out = a.c_group > 0 ? (a.M / a.c_group) * (a.c_group - a.c_drop) : a.M;
    TcParams p{a.M, a.N, a.K, a.bias, a.C, a.ldc, a.epi, a.alpha, a.out_type, fmt, 0, a.c_group, a.c_drop, a.C0, m_out, a.w_dynamic};
    const int tiles_n = (a.N + BN - 1) / BN, tiles_m = (a.M + 2 * BM - 1) / (2 * BM), splits = a.splits > 1 ? a.splits : 1;
    int dev = 0, sms = 148;
    cudaGetDevice(&dev); cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const int npairs = std::min(tiles_n * tiles_m * splits, sms / 2);
    launch_k_cluster(gemm_tc_pair256_persist_kernel<BN, STAGES>, dim3(2 * npairs), dim3(TC_THREADS), smem, st, 2, tmA, tmB, p, tiles_n, tiles_m, splits);
}
void launch_pair256_persist(const GemmArgs& a, int fmt, int bn, cudaStream_t st) {
    switch (bn) {                                                   // stages: what fits next to the 18 KB epilogue patch in 227 KB
        case 256: launch_cfg_pair256_persist<256, 6>(a, fmt, st); break;
        case 208: launch_cfg_pair256_persist<208, 6>(a, fmt, st); break;
        case 160: launch_cfg_pair256_persist<160, 7>(a, fmt, st); break;
        case 128: launch_cfg_pair256_persist<128, 8>(a, fmt, st); break;
        case 112: launch_cfg_pair256_persist<112, 8>(a, fmt, st); break;
        default: throw CudaError("gemm_tc: persistent pair256 tile not instantiated");
    }
}
// Pair tiles for large batches: BN per shape so that the pair tiles fill whole waves of the 74 SM pairs. Per-SM cost of a tile
// ~ the bytes it stages per k-block, (128 + BN/2) rows (+ a fixed share for prologue / epilogue that does not overlap).
int pick_pair256_bn(int M, int N) {
    // Measured (profiles/r01_gemm_large_*.txt): a pair tile's main loop is latency-bound on its own (3-4 stages of ~25 KB against
    // ~1.5 us of L2 -> SM latency under load), so what pays is many tiles with two co-resident CTAs per SM: the SMALLEST BN whose
    // pair tiles still fit the 148 co-resident pair slots (74 SM pairs x 2). Not worth it when even BN = 112 leaves the machine
    // short of tiles (returns 0: the single-CTA tiles win there).
    const int tiles_m = (M + 2 * BM - 1) / (2 * BM);
    auto tiles = [&](int bn) { return (long long)tiles_m * ((N + bn - 1) / bn); };
    static const int min_pairs = [] { const char* e = getenv("NSB_PAIR256_MIN_PAIRS"); return e ? atoi(e) : 100; }();
    if (tiles(112) < min_pairs) return 0;
    for (int bn : {112, 160, 208, 256}) if (tiles(bn) <= 148) return bn;
    int best = 256; long long best_cost = 0;
    for (int bn : {256, 208, 160, 112}) {
        const long long cost = ((tiles(bn) + 147) / 148) * (BM + bn / 2);
        if (!best_cost || cost < best_cost) { best = bn; best_cost = cost; }
    }
    return best;
}
// the same choice for the fused Q8_0 / Q4_0 pair tiles (BN <= 208: raw + dequantised half tiles and two CTAs per SM)
int pick_q8_pair256_bn(int M, int N) {
    const int tiles_m = (M + 2 * BM - 1) / (2 * BM);
    auto tiles = [&](int bn) { return (long long)tiles_m * ((N + bn - 1) / bn); };
    if (tiles(112) < 100) return 0;
    for (int bn : {112, 160, 208}) if (tiles(bn) <= 148) return bn;
    int best = 208; long long best_cost = 0;
    for (int bn : {208, 160, 112}) {
        const long long cost = ((tiles(bn) + 147) / 148) * (BM + bn / 2);
        if (!best_cost || cost < best_cost) { best = bn; best_cost = cost; }
    }
    return best;
}
void launch_pair256(const GemmArgs& a, int fmt, int bn, cudaStream_t st) {
    switch (bn) {
        case 256: launch_cfg_pair256<256, 3>(a, fmt, st); break;
        case 208: launch_cfg_pair256<208, 3>(a, fmt, st); break;
        case 160: launch_cfg_pair256<160, 4>(a, fmt, st); break;
        case 112: launch_cfg_pair256<112, 4>(a, fmt, st); break;
        default: throw CudaError("gemm_tc: pair256 tile not instantiated");
    }
}

// A forced tile config (nsb_bench_gemm, nsb_op_gemm_ex) must name a tile the dispatch below instantiates for this operand type, and the
// tile's grid must cover all N columns; anything else is the caller's error, not a launch that computes part of C.
void check_forced_config(const GemmArgs& a, int fmt) {
    const int bn = a.force_bn, st = a.force_stages;
    auto fail = [&](const char* why) {
        throw std::invalid_argument("gemm_tc: forced tile " + std::to_string(bn) + "/" + std::to_string(st) + ": " + why);
    };
    auto one_of = [](int v, std::initializer_list<int> l) { return std::find(l.begin(), l.end(), v) != l.end(); };
    if (a.w_scales) {                                             // fused Q8_0 / Q4_0 planes: only the 256-row pair tiles (grid rounds up along N)
        if (st != 95 || !one_of(bn, {112, 160, 208})) fail("not instantiated for Q8_0 / Q4_0 planes");
        return;
    }
    if (st == 95) fail("the fused Q8_0 tiles need Q8_0 / Q4_0 planes");
    if (st == 96 || st == 97) {                                   // 256-row pair tiles: grid rounds up along N, the epilogue clips the last tile
        if (fmt == 2) fail("pair tiles are 16-bit only");
        if (!one_of(bn, st == 97 ? std::initializer_list<int>{112, 160, 208, 256} : std::initializer_list<int>{112, 128, 160, 208, 256})) fail("not instantiated");
        return;
    }
    const int key = bn * 100 + st;
    if (!one_of(key, {3204, 3205, 3208, 6404, 6498, 6406, 12803, 12804, 25602, 25603})) fail("not instantiated");
    if (fmt == 2 && !one_of(key, {3205, 6404, 12803, 12804, 25602})) fail("not instantiated for tf32");
    if (a.N % bn != 0) fail("the grid does not cover N");
}
void check_splits(const GemmArgs& a, int BK) {
    if (a.splits > 1 && (a.epi != EPI_PARTIAL || (a.K / BK) % a.splits != 0))
        throw std::invalid_argument("gemm_tc: bad split-K request (" + std::to_string(a.splits) + " slices of " + std::to_string(a.K / BK) + " k-blocks)");
}

template <int BN, int STAGES, int EB>
void launch_cfg_e(const GemmArgs& a, int fmt, cudaStream_t st) {
    if (a.multicast && multicast_enabled() && (a.N / BN) % 4 == 0) launch_cfg_c<BN, STAGES, EB, 4>(a, fmt, st);
    else launch_cfg_c<BN, STAGES, EB, 1>(a, fmt, st);
}
template <int BN, int STAGES>
void launch_cfg(const GemmArgs& a, int fmt, cudaStream_t st) {
    if (fmt == 2) {
        if constexpr ((BN == 32 && STAGES == 5) || (BN == 64 && STAGES == 4) || (BN == 128 && (STAGES == 3 || STAGES == 4)) || (BN == 256 && STAGES == 2))
            launch_cfg_e<BN, STAGES, 4>(a, fmt, st);
        else throw CudaError("gemm_tc: tile config not instantiated for tf32");
    } else launch_cfg_e<BN, STAGES, 2>(a, fmt, st);
}
}  // namespace

// Q8_0 planes -> fp16 [N][K], once per GEMM launch, for batches of many 128-row tiles: there every m-tile CTA of the fused
// kernel repeats the dequantisation of the same weight tile (14x at 1792 rows) and the dequant warps, not HBM, set the pace.
// The 2-8 MB fp16 copy is consumed by the next kernel straight out of L2; HBM still only sees the int8 + scale planes.
// Same arithmetic as the fused path (fp16(d) * q, one rounding): bit-identical operand values.
namespace {
__global__ void __launch_bounds__(256) dequant_q8_kernel(const uint4* __restrict__ q, const __half* __restrict__ sc, uint4* __restrict__ out,
                                                         size_t n_vec, int K) {
    NSB_KERNEL_PROLOGUE(TR_OTHER)                                                 // the scratch may still be read by the previous GEMM
    const __half2 off = __floats2half2_rn(1152.0f, 1152.0f);
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_vec; i += (size_t)gridDim.x * blockDim.x) {
        const uint4 raw = q[i];
        const size_t e0 = i * 16, row = e0 / (size_t)K, col = e0 % (size_t)K;
        const __half2 d2 = __half2half2(sc[row * (size_t)(K / 32) + col / 32]);
        const uint32_t w4[4] = {raw.x, raw.y, raw.z, raw.w};
        __half2 h[8];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const uint32_t x = w4[j] ^ 0x80808080u;
            const uint32_t lo = __byte_perm(x, 0x64646464u, 0x5140), hi = __byte_perm(x, 0x64646464u, 0x5342);
            h[2 * j] = __hmul2(__hsub2(*reinterpret_cast<const __half2*>(&lo), off), d2);
            h[2 * j + 1] = __hmul2(__hsub2(*reinterpret_cast<const __half2*>(&hi), off), d2);
        }
        out[2 * i] = *reinterpret_cast<uint4*>(&h[0]);
        out[2 * i + 1] = *reinterpret_cast<uint4*>(&h[4]);
    }
    NSB_KERNEL_EPILOGUE();
}
}  // namespace
namespace {
// Q4_0 nibble plane [N][K / 2] + scales -> fp16 [N][K]: one thread per 32-value block (16 bytes in, 64 bytes out)
__global__ void __launch_bounds__(256) dequant_q4_kernel(const uint4* __restrict__ q, const __half* __restrict__ sc, uint4* __restrict__ out, size_t nb) {
    NSB_KERNEL_PROLOGUE(TR_OTHER)
    const __half2 off = __floats2half2_rn(1032.0f, 1032.0f);
    for (size_t b = (size_t)blockIdx.x * blockDim.x + threadIdx.x; b < nb; b += (size_t)gridDim.x * blockDim.x) {
        const uint4 raw = q[b];
        const __half2 d2 = __half2half2(sc[b]);
        const uint32_t w4[4] = {raw.x, raw.y, raw.z, raw.w};
#pragma unroll
        for (int half = 0; half < 2; ++half) {                                   // values 0..15 = low nibbles, 16..31 = high nibbles
            __half2 h[8];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const uint32_t x = (w4[j] >> (4 * half)) & 0x0F0F0F0Fu;
                const uint32_t lo = __byte_perm(x, 0x64646464u, 0x5140), hi = __byte_perm(x, 0x64646464u, 0x5342);
                h[2 * j] = __hmul2(__hsub2(*reinterpret_cast<const __half2*>(&lo), off), d2);
                h[2 * j + 1] = __hmul2(__hsub2(*reinterpret_cast<const __half2*>(&hi), off), d2);
            }
            out[4 * b + 2 * half] = *reinterpret_cast<uint4*>(&h[0]);
            out[4 * b + 2 * half + 1] = *reinterpret_cast<uint4*>(&h[4]);
        }
    }
    NSB_KERNEL_EPILOGUE();
}
}  // namespace
void launch_dequant_q8(const void* q, const void* scales, void* out_f16, int N, int K, cudaStream_t st, int q4) {
    if (K % 32 != 0) throw CudaError("dequant_q8: K must be a multiple of 32");
    if (q4) {
        const size_t nb = (size_t)N * K / 32;
        launch_k(dequant_q4_kernel, dim3((unsigned)std::min<size_t>((nb + 255) / 256, 148 * 8)), dim3(256), 0, st, (const uint4*)q, (const __half*)scales, (uint4*)out_f16, nb);
        return;
    }
    const size_t n_vec = (size_t)N * K / 16;
    const int blocks = (int)std::min<size_t>((n_vec + 255) / 256, 148 * 8);
    launch_k(dequant_q8_kernel, dim3(blocks), dim3(256), 0, st, (const uint4*)q, (const __half*)scales, (uint4*)out_f16, n_vec, K);
}

// in_type: OUT_F16 / OUT_BF16 / OUT_F32 (= tf32) -- type of A and W. Requires K % 64 == 0 (tf32: 32), N % 32 == 0, 16-byte aligned rows.
void launch_gemm_tc(const GemmArgs& a, int in_type, cudaStream_t st) {
    if (a.M <= 0) return;
    if (a.group != 0) throw CudaError("gemm_tc: row maps are not supported");
    const int fmt = in_type == OUT_F32 ? 2 : in_type == OUT_BF16 ? 1 : 0;
    const int BK = fmt == 2 ? 32 : 64;
    if (a.K % BK != 0 || a.N % 32 != 0 || (a.lda % (fmt == 2 ? 4 : 8)) != 0 || (a.ldc % 4) != 0)
        throw CudaError("gemm_tc: unsupported shape (need K % 64 == 0 (tf32: 32), N % 32 == 0, 16-byte aligned rows)");
    if (a.c_group > 0 && a.M % a.c_group != 0) throw CudaError("gemm_tc: M must be a multiple of the output row group");
    if (a.a_fold && (fmt != 2 || a.K != 3 * a.a_fold || a.a_fold % BK != 0)) throw CudaError("gemm_tc: 3xTF32 needs fp32 operands and K = 3 x the folded width");
    const int tiles_m = (a.M + BM - 1) / BM;
    if (a.w_scales) {                                             // Q8_0 planes: fused-dequant kernel (A is fp16)
        if (fmt != 0) throw CudaError("gemm_q8: activations must be fp16");
        check_splits(a, BK);
        if (a.force_bn) { check_forced_config(a, fmt); launch_q8_pair256(a, a.force_bn, st); return; }      // tuning hook
        if (tiles_m >= pair256_min_tiles() && q8_pair256_enabled()) {   // large batches: fused dequantisation on the 256-row CTA-pair tiles
            static const int split_bn = [] { const char* e = getenv("NSB_SPLIT_BN"); return e ? atoi(e) : 112; }();
            const int bn = a.splits > 1 ? (split_bn == 256 ? 208 : split_bn) : pick_q8_pair256_bn(a.M, a.N);
            if (bn) { launch_q8_pair256(a, bn, st); return; }
        }
        if (a.splits > 1) { if (a.N % 64 == 0 && a.K >= 4096) launch_cfg_q8<64, 4>(a, st); else launch_cfg_q8<32, 5>(a, st); return; }
        if (a.N % 128 == 0 && (long long)tiles_m * (a.N / 128) >= 120) launch_cfg_q8<128, 4>(a, st);
        else if (a.N % 64 == 0 && (long long)tiles_m * (a.N / 64) >= 120) launch_cfg_q8<64, 4>(a, st);
        else launch_cfg_q8<32, 5>(a, st);
        return;
    }
    if (a.force_bn) {                                             // tuning hook
        check_splits(a, BK);
        check_forced_config(a, fmt);
        if (a.force_stages == 97) { launch_pair256(a, fmt, a.force_bn, st); return; }
        if (a.force_stages == 96) { launch_pair256_persist(a, fmt, a.force_bn, st); return; }
        const int key = a.force_bn * 100 + a.force_stages;
        switch (key) {
            case 3204: launch_cfg<32, 4>(a, fmt, st); break;
            case 3205: launch_cfg<32, 5>(a, fmt, st); break;
            case 3208: launch_cfg<32, 8>(a, fmt, st); break;
            case 6404: launch_cfg<64, 4>(a, fmt, st); break;
            case 6498: launch_cfg_pair<64, 8>(a, fmt, st); break;
            case 6406: launch_cfg<64, 6>(a, fmt, st); break;
            case 12803: launch_cfg<128, 3>(a, fmt, st); break;
            case 12804: launch_cfg<128, 4>(a, fmt, st); break;
            case 25602: launch_cfg<256, 2>(a, fmt, st); break;
            case 25603: launch_cfg<256, 3>(a, fmt, st); break;
            default: throw CudaError("gemm_tc: tile config not instantiated");
        }
        return;
    }
    if (a.splits > 1) {
        check_splits(a, BK);
        if (fmt != 2 && tiles_m >= 8 && pair256_enabled()) {            // large-batch split-K (FFN down): wide pair tiles
            static const int bn = [] { const char* e = getenv("NSB_SPLIT_BN"); return e ? atoi(e) : 112; }();
            if (pair256_persist_enabled()) launch_pair256_persist(a, fmt, bn, st); else launch_pair256(a, fmt, bn, st);
            return;
        }
        if (a.N % 128 == 0 && a.M > 128 && fmt == 2) { launch_cfg<128, 4>(a, fmt, st); return; }
        if (a.N % 64 == 0 && a.K >= 4096) launch_cfg<64, 4>(a, fmt, st); else launch_cfg<32, 5>(a, fmt, st);
        return;
    }
    // Tile choice (profiles/r01_gemm_tile_sweep*.txt). Small batches stream weights: narrow tiles so that >= ~1 wave of CTAs pulls.
    // Large batches are tensor-bound: wide tiles, and a shared-memory footprint <= ~100 KB so that two CTAs share an SM and one's
    // epilogue overlaps the other's main loop (the kernel has a single TMEM accumulator per CTA).
    // single 128-row tile, 16-bit operands: CTA-pair tiles (8 stages; 12 / 16 measured slower in the step: the main loop does not
    // speed up and the next kernel loses its early residency, profiles/r01_notes.md)
    if (fmt != 2 && a.pair && !a.w_dynamic && pair_gemm_enabled() && tiles_m == 1 && a.N % 64 == 0) { launch_cfg_pair<64, 8>(a, fmt, st); return; }
    // >= 4 row tiles, 16-bit operands: 256-row CTA-pair tiles (the single-CTA tile is L2 -> SM ingest bound there)
    // (the small square matrices -- attention out-projection, pointwise-2 -- measured 7.8 us on 128 x 128 single-CTA tiles against 9.0 us
    //  on the best pair tile at 1792 rows with a plain store epilogue, profiles/r02_gemm_sweep.txt, but no faster with the residual
    //  read-modify-write epilogue they run with in the step: left on the pair tiles)
    if (fmt != 2 && tiles_m >= pair256_min_tiles() && pair256_enabled()) {
        const int bn = pick_pair256_bn(a.M, a.N);
        if (bn) { if (pair256_persist_enabled()) launch_pair256_persist(a, fmt, bn, st); else launch_pair256(a, fmt, bn, st); return; }
    }
    const long long t256 = a.N % 256 == 0 ? (long long)tiles_m * (a.N / 256) : 0, t128 = a.N % 128 == 0 ? (long long)tiles_m * (a.N / 128) : 0;
    if (t256 >= 200) launch_cfg<256, 2>(a, fmt, st);
    else if (t128 >= 200) launch_cfg<128, 3>(a, fmt, st);
    else if (t128 >= 100) launch_cfg<128, 4>(a, fmt, st);
    else if (a.N % 64 == 0 && (long long)tiles_m * (a.N / 64) >= 120) launch_cfg<64, 4>(a, fmt, st);
    else launch_cfg<32, 5>(a, fmt, st);
}

}  // namespace nsb
