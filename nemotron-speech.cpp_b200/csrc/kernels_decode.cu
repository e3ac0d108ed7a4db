// kernels_decode.cu -- batched RNN-T greedy decode as ONE persistent kernel (sm_100a), one CTA per SM.
//
// Reference behaviour being replaced: decode_one_step + the per-frame loop of process_mel_chunk_streaming
// (src/nemo-stream.cpp:788-878, :1035-1047) on top of build_decoder_step / build_lstm_cell / build_joint
// (src/nemo-ggml.cpp:503-542, :1013-1100). The reference launches one graph and does 6-8 host<->device
// copies PER SYMBOL PER STREAM; here all streams of a step are decoded by one launch with no host round-trips.
//
// Semantics kept exactly (nemo-stream.cpp:813-875): up to 10 symbols per encoder frame; argmax = lowest index
// among maxima; blank => next frame, LSTM state untouched; non-blank => emit, prev_token = token, commit h', c'.
// The reference re-runs the LSTM for every evaluation and throws the result away on blank; since
// (prev_token, h, c) only change on emission the candidate (h', c', joint.pred projection) is kept per stream and
// recomputed only after an emission -- arithmetic-identical.
//
// Structure. The grid advances in "rounds": one joint evaluation for every still-active stream, preceded by the
// prediction network for the streams that emitted in the previous round. Every phase is a skinny fp32 GEMM
//     OUT[stream][row] = sum_k X[stream][k] * W[row][k]          (streams <= 64 per block, K = 1280 or 640)
// split over the grid by weight rows, so each weight byte is pulled from L2 once per round and stream block. Inside
// a CTA the 8 warps split K; every warp copies ITS k-slice of the weight rows and of the stream vectors into a private
// shared-memory region with one burst of 16-byte cp.async (all requests in flight at once: one L2 latency per item,
// no block-wide barrier), then a lane accumulates an RPL x SPL (rows x streams) register tile out of shared memory
// (padded rows: conflict-free, W broadcast over the 8 stream groups, X over the 4 row groups); partial tiles of the
// 8 warps meet in shared memory.
//   * per-stream control state (frame index, symbols at this frame, parity of the committed LSTM buffer, previous
//     token) is REPLICATED in every CTA's shared memory and advanced identically from the broadcast argmax keys, so
//     a round costs 4 grid barriers with the prediction network and 1 without;
//   * the argmax across row slices is one 64-bit atomicMax per (CTA, stream): key = orderable(logit) << 32 | ~index
//     (largest logit wins, ties go to the lowest index = "first max wins");
//   * h/c are double-buffered per stream: the candidate is written to the other parity, committing = flipping the
//     parity bit (no copy, no extra barrier);
//   * the grid barrier is a monotonic counter in HBM (arrive = one atomicAdd, wait = ld.acquire spin, bounded).
#include <algorithm>
#include <cstdlib>

#include "kernels.cuh"

namespace nsb {

NSB_DEFINE_TRACE_BINDER(trace_bind_decode)

namespace {
constexpr int NT = 256, NW = NT / 32;
constexpr int RSTR = 40;             // padded stream stride of the partial-tile buffers
constexpr int RC_MAX = 20;           // weight rows per work item: 20 (LSTM: 5 units x 4 gates) or 8 (pred, joint)
constexpr int MAXB = 1024;           // max streams per step
constexpr int PAR_STRIDE = 2 * HID;  // one parity copy of (layer 0 | layer 1) h or c
// per-warp staging region (floats): LSTM 20 rows + 16 streams of 160+4; joint 8 rows + 2 x 32 streams of 80+4
constexpr int STAGE_FLOATS = 8 * 84 + 2 * 32 * 84;
static_assert(STAGE_FLOATS >= (20 + 16) * 164, "staging region too small for the LSTM phase");

struct DecSmem {
    float stage[NW][STAGE_FLOATS];   // phase(): per-warp W / X slices, reused for the warp's partial tile; phase_pipe(): one flat ring of stages
    unsigned long long keys[NW][32]; // phase_pipe() joint: per-warp argmax keys of a tile
    float sums[RC_MAX][RSTR];
    int slot[MAXB], prev[MAXB], list[MAXB];
    short fi[MAXB], oc[MAXB];        // frame index within the chunk, tokens emitted this step
    unsigned char sc[MAXB], need[MAXB], par[MAXB];   // symbols at this frame, candidate stale, committed parity
    int warp_cnt[NW];
};

__device__ __forceinline__ void cp_async16(float* smem_dst, const float* gsrc) {                     // L2 -> smem, bypasses L1
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() {
    asm volatile("cp.async.commit_group;" ::: "memory");
    asm volatile("cp.async.wait_group 0;" ::: "memory");
}
__device__ __forceinline__ unsigned ld_acquire(const unsigned* p) {
    unsigned v; asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory"); return v;
}

// grid-wide barrier: every CTA is resident (cooperative launch, one CTA per SM)
__device__ __forceinline__ void grid_barrier(unsigned* ctr, unsigned& epoch, unsigned nblk) {
    __syncthreads();
    if (threadIdx.x == 0) {
        epoch += 1;
        const unsigned target = epoch * nblk;
        // release-arrive (orders every write of this CTA made before the bar.sync above), acquire-spin
        asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(ctr) : "memory");
        unsigned it = 0;
        while (ld_acquire(ctr) < target) { if (++it > (1u << 26)) __trap(); }     // a protocol bug traps instead of hanging the GPU
    }
    __syncthreads();
}

__device__ __forceinline__ unsigned long long argmax_key(float v, int idx) {
    unsigned u = __float_as_uint(v);
    u = (u & 0x80000000u) ? ~u : (u | 0x80000000u);                              // monotone float -> uint
    return ((unsigned long long)u << 32) | (unsigned long long)(0xFFFFFFFFu - (unsigned)idx);
}

// block-wide stable compaction of {b : pred(b)} into sm.list; returns the count (block-uniform)
template <class Pred>
__device__ int compact(DecSmem& sm, int B, Pred pred) {
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    int base = 0;
    for (int b0 = 0; b0 < B; b0 += NT) {
        const int b = b0 + tid;
        const bool f = b < B && pred(b);
        const unsigned m = __ballot_sync(0xffffffffu, f);
        if (lane == 0) sm.warp_cnt[warp] = __popc(m);
        __syncthreads();
        int off = base, tot = 0;
        for (int w = 0; w < NW; ++w) { if (w < warp) off += sm.warp_cnt[w]; tot += sm.warp_cnt[w]; }
        if (f) sm.list[off + __popc(m & ((1u << lane) - 1))] = b;
        base += tot;
        __syncthreads();
    }
    return base;
}

enum { MODE_LSTM = 0, MODE_PRED = 1, MODE_JOINT = 2 };

// One phase over the n listed streams, in blocks of SB = 8 * SPL streams. RPL rows x SPL streams per lane;
// 4 row groups x 8 stream groups per warp.
template <int RPL, int SPL, int MODE>
__device__ void phase(const DecodeArgs& a, DecSmem& sm, int layer, int n, int round, int ne0) {
    constexpr int RC = 4 * RPL, SB = 8 * SPL;
    constexpr int K = MODE == MODE_LSTM ? 2 * HID : HID;
    constexpr int KW = K / NW;                                                    // k-slice of one warp (160 or 80)
    constexpr int WS = KW + 4, VPR = KW / 4;                                      // padded smem row stride; 16-byte vectors per row slice
    static_assert((RC + (MODE == MODE_JOINT ? 2 : 1) * SB) * WS <= STAGE_FLOATS, "staging region overflow");
    const int n_chunks = MODE == MODE_LSTM ? HID / RPL : MODE == MODE_PRED ? JOINT / RC : (VOCAB + RC - 1) / RC;
    const int n_sblk = (n + SB - 1) / SB;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, rg = lane >> 3, sg = lane & 7;
    const int kbeg = warp * KW;
    const bool second_half = MODE == MODE_LSTM && kbeg >= HID;                    // LSTM: k < 640 is the input, k >= 640 the recurrent part
    const int koff = second_half ? kbeg - HID : kbeg;
    float* wsm = sm.stage[warp];
    float* xsm = wsm + RC * WS;
    float* dsm = xsm + SB * WS;                                                   // joint only

    for (int item = blockIdx.x; item < n_chunks * n_sblk; item += gridDim.x) {
        const int chunk = item % n_chunks, s0 = (item / n_chunks) * SB, ns = min(SB, n - s0);
        // ---- stage this warp's k-slice: weight rows, then the stream vectors ----
        for (int p = lane; p < RC * VPR; p += 32) {
            const int r = p / VPR, c = (p % VPR) * 4;
            const float* src;
            if (MODE == MODE_LSTM) {                                              // row group = gate (i,f,g,o), RPL units per chunk
                const int row = (r / RPL) * HID + chunk * RPL + (r % RPL);
                src = (second_half ? a.w.w_hh[layer] : a.w.w_ih[layer]) + (size_t)row * HID + koff + c;
            } else if (MODE == MODE_PRED) {
                src = a.w.pred_w + (size_t)(chunk * RC + r) * HID + koff + c;
            } else {
                src = a.w.out_w + (size_t)min(chunk * RC + r, VOCAB - 1) * JOINT + koff + c;
            }
            cp_async16(wsm + r * WS + c, src);
        }
        for (int p = lane; p < ns * VPR; p += 32) {
            const int g = p / VPR, c = (p % VPR) * 4;
            const int b = sm.list[s0 + g], slot = sm.slot[b], par = sm.par[b];
            const float* hb = a.s.hbuf + (size_t)slot * 2 * PAR_STRIDE;
            const float* src;
            if (MODE == MODE_LSTM) {
                if (layer == 0) src = second_half ? hb + par * PAR_STRIDE                                   // h0 (committed)
                                                  : a.w.embed + (size_t)sm.prev[b] * HID;                   // nemo-stream.cpp:825-828
                else src = second_half ? hb + par * PAR_STRIDE + HID                                        // h1 (committed)
                                       : hb + (par ^ 1) * PAR_STRIDE;                                       // layer-1 input = layer-0 h'
            } else if (MODE == MODE_PRED) {
                src = hb + (par ^ 1) * PAR_STRIDE + HID;                                                    // candidate decoder output
            } else {
                src = a.enc_proj + ((size_t)b * a.T + sm.fi[b]) * JOINT;
                cp_async16(dsm + g * WS + c, a.s.dec_proj + (size_t)slot * JOINT + koff + c);
            }
            cp_async16(xsm + g * WS + c, src + koff + c);
        }
        cp_async_wait_all();
        __syncwarp();

        float acc[RPL][SPL];
#pragma unroll
        for (int i = 0; i < RPL; ++i)
#pragma unroll
            for (int j = 0; j < SPL; ++j) acc[i][j] = 0.f;
#pragma unroll 4
        for (int k = 0; k < KW; k += 4) {
            float4 w[RPL], x[SPL];
#pragma unroll
            for (int i = 0; i < RPL; ++i) w[i] = *reinterpret_cast<const float4*>(wsm + (rg * RPL + i) * WS + k);
#pragma unroll
            for (int j = 0; j < SPL; ++j) {
                x[j] = *reinterpret_cast<const float4*>(xsm + (sg + 8 * j) * WS + k);
                if (MODE == MODE_JOINT) {                                         // z = relu(enc_proj + pred_proj)  (nemo-ggml.cpp:1092-1094)
                    const float4 d = *reinterpret_cast<const float4*>(dsm + (sg + 8 * j) * WS + k);
                    x[j].x = fmaxf(x[j].x + d.x, 0.f); x[j].y = fmaxf(x[j].y + d.y, 0.f);
                    x[j].z = fmaxf(x[j].z + d.z, 0.f); x[j].w = fmaxf(x[j].w + d.w, 0.f);
                }
            }
#pragma unroll
            for (int i = 0; i < RPL; ++i)
#pragma unroll
                for (int j = 0; j < SPL; ++j) {
                    acc[i][j] = fmaf(w[i].x, x[j].x, acc[i][j]); acc[i][j] = fmaf(w[i].y, x[j].y, acc[i][j]);
                    acc[i][j] = fmaf(w[i].z, x[j].z, acc[i][j]); acc[i][j] = fmaf(w[i].w, x[j].w, acc[i][j]);
                }
        }
        __syncwarp();                                                             // the warp's partial tile reuses its own staging region
        float* red = sm.stage[warp];
#pragma unroll
        for (int i = 0; i < RPL; ++i)
#pragma unroll
            for (int j = 0; j < SPL; ++j) red[(rg * RPL + i) * RSTR + sg + 8 * j] = acc[i][j];
        __syncthreads();
        for (int e = tid; e < RC * ns; e += NT) {                                 // fixed warp order => deterministic sums
            const int rr = e / ns, g = e % ns;
            float s = sm.stage[0][rr * RSTR + g];
#pragma unroll
            for (int w8 = 1; w8 < NW; ++w8) s += sm.stage[w8][rr * RSTR + g];
            sm.sums[rr][g] = s;
        }
        __syncthreads();
        if (MODE == MODE_LSTM) {                                                  // gate order i,f,g,o (nemo-ggml.cpp:518-541)
            for (int e = tid; e < RPL * ns; e += NT) {
                const int uu = e / ns, g = e % ns, b = sm.list[s0 + g], slot = sm.slot[b], par = sm.par[b];
                const int u = chunk * RPL + uu;
                float gate[4];
#pragma unroll
                for (int q = 0; q < 4; ++q)
                    gate[q] = (sm.sums[q * RPL + uu][g] + __ldg(a.w.b_ih[layer] + q * HID + u)) + __ldg(a.w.b_hh[layer] + q * HID + u);
                const float ig = sigmoid_exact(gate[0]), fg = sigmoid_exact(gate[1]), gg = tanhf(gate[2]), og = sigmoid_exact(gate[3]);
                const size_t o_old = (size_t)slot * 2 * PAR_STRIDE + par * PAR_STRIDE + layer * HID + u;
                const size_t o_new = (size_t)slot * 2 * PAR_STRIDE + (par ^ 1) * PAR_STRIDE + layer * HID + u;
                const float cn = fg * __ldcg(a.s.cbuf + o_old) + ig * gg;
                a.s.cbuf[o_new] = cn; a.s.hbuf[o_new] = og * tanhf(cn);
            }
        } else if (MODE == MODE_PRED) {                                           // joint.pred (nemo-ggml.cpp:1086-1087)
            for (int e = tid; e < RC * ns; e += NT) {
                const int rr = e / ns, g = e % ns, j = chunk * RC + rr;
                a.s.dec_proj[(size_t)sm.slot[sm.list[s0 + g]] * JOINT + j] = sm.sums[rr][g] + __ldg(a.w.pred_b + j);
            }
        } else {                                                                  // logits of this row slice -> argmax key
            if (tid < ns) {
                const int b = sm.list[s0 + tid];
                float bv = -INFINITY; int bi = 0;
#pragma unroll
                for (int rr = 0; rr < RC; ++rr) {
                    const int v = chunk * RC + rr;
                    if (v < VOCAB) {
                        const float s = sm.sums[rr][tid] + __ldg(a.w.out_b + v);
                        if (s > bv) { bv = s; bi = v; }                           // ascending v, strict > : first max wins (:847-854)
                        if (a.logits_tap && b == 0 && ne0 < a.logits_tap_cap) a.logits_tap[(size_t)ne0 * VOCAB + v] = s;
                    }
                }
                atomicMax(a.best + (size_t)(round % 3) * a.B + b, argmax_key(bv, bi));
            }
        }
        __syncthreads();                                                          // staging regions / sums are reused by the next item
    }
}


// ------------------------------------------------------------------------------------------
// phase_pipe(): the same three skinny GEMMs as phase(), organised as a CTA-tiled SIMT GEMM behind a multi-stage cp.async ring.
// phase() stages ONE item (a row slab x a stream block) per round trip to L2, which is fine when a CTA has one or two items per
// phase (148 CTAs, a handful of streams) and poor otherwise: on a narrow grid (decode overlap: ~20 CTAs walk 8 items per phase) and
// at large batches (many stream blocks per row slab) every item exposes its own L2 latency. Here the CTA walks a flat sequence of
// (item, K chunk) steps; the loads of step q + NST - 1 are issued while step q is computed, across item boundaries, so L2 -> SM
// streaming never stops inside a phase.
//   tile: RT = 32 RPL weight rows x ST = 8 SPL streams; 8 warps x (4 row groups x 8 stream groups) lanes, RPL x SPL outputs per lane;
//         LSTM: row group = gate (i, f, g, o), a warp owns RPL hidden units, the four gate sums of a unit meet by shuffle.
//   K in 8 chunks (160 or 80 wide): chunk partial sums are formed from zero and added in chunk order -- exactly the summation order
//   of phase() (its 8 warps own the same 8 K slices and are summed in warp order), so both paths, any grid size, give the same bits.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned long long shfl_xor_u64(unsigned long long v, int m) {
    const unsigned lo = __shfl_xor_sync(0xffffffffu, (unsigned)v, m), hi = __shfl_xor_sync(0xffffffffu, (unsigned)(v >> 32), m);
    return ((unsigned long long)hi << 32) | lo;
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

template <int RPL, int SPL, int MODE>
__device__ void phase_pipe(const DecodeArgs& a, DecSmem& sm, int layer, int n, int round, int ne0) {
    constexpr int K = MODE == MODE_LSTM ? 2 * HID : HID, NCH = 8, KW = K / NCH, WS = KW + 4, VPR = KW / 4;
    constexpr int RT = 32 * RPL, ST = 8 * SPL, XM = MODE == MODE_JOINT ? 2 : 1;
    constexpr int STAGE_F = (RT + XM * ST) * WS;
    constexpr int NST_FIT = NW * STAGE_FLOATS / STAGE_F, NST = NST_FIT > 6 ? 6 : NST_FIT;
    static_assert(NST >= 3, "at least three stages in the ring");
    const int rows_total = MODE == MODE_LSTM ? 4 * HID : MODE == MODE_PRED ? JOINT : VOCAB;
    const int n_rt = (rows_total + RT - 1) / RT, n_sb = (n + ST - 1) / ST, n_items = n_rt * n_sb;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, rg = lane >> 3, sg = lane & 7;
    const int my_items = (int)blockIdx.x < n_items ? (n_items - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;
    const int total_steps = my_items * NCH;
    float* ring = &sm.stage[0][0];

    // global row of tile row rr (LSTM: rr = warp (4 RPL) + gate RPL + i  <->  row gate * 640 + unit)
    auto w_row = [&](int rt, int rr) -> int {
        if (MODE == MODE_LSTM) { const int w = rr / (4 * RPL), q = (rr / RPL) & 3, i = rr % RPL; return q * HID + rt * (8 * RPL) + w * RPL + i; }
        return min(rt * RT + rr, rows_total - 1);
    };
    auto issue = [&](int q) {
        if (q < total_steps) {
            const int item = (int)blockIdx.x + (q / NCH) * (int)gridDim.x, c = q % NCH;
            const int rt = item % n_rt, s0 = (item / n_rt) * ST, ns = min(ST, n - s0);
            float* st = ring + (q % NST) * STAGE_F;
            for (int p = tid; p < RT * VPR; p += NT) {
                const int rr = p / VPR, v = (p % VPR) * 4, row = w_row(rt, rr);
                const float* src;
                if (MODE == MODE_LSTM) src = (c < NCH / 2 ? a.w.w_ih[layer] : a.w.w_hh[layer]) + (size_t)row * HID + (c % (NCH / 2)) * KW + v;   // k < 640: input, k >= 640: recurrent
                else src = (MODE == MODE_PRED ? a.w.pred_w : a.w.out_w) + (size_t)row * HID + c * KW + v;
                cp_async16(st + rr * WS + v, src);
            }
            for (int p = tid; p < ns * VPR; p += NT) {
                const int g = p / VPR, v = (p % VPR) * 4;
                const int b = sm.list[s0 + g], slot = sm.slot[b], par = sm.par[b];
                const float* hb = a.s.hbuf + (size_t)slot * 2 * PAR_STRIDE;
                const float* src;
                if (MODE == MODE_LSTM) {
                    const int kc = (c % (NCH / 2)) * KW;
                    if (c < NCH / 2) src = (layer == 0 ? a.w.embed + (size_t)sm.prev[b] * HID : hb + (par ^ 1) * PAR_STRIDE) + kc;      // nemo-stream.cpp:825-828 | layer-0 h'
                    else src = hb + par * PAR_STRIDE + layer * HID + kc;                                                               // committed h of this layer
                } else if (MODE == MODE_PRED) {
                    src = hb + (par ^ 1) * PAR_STRIDE + HID + c * KW;                                                                   // candidate decoder output
                } else {
                    src = a.enc_proj + ((size_t)b * a.T + sm.fi[b]) * JOINT + c * KW;
                    cp_async16(st + (RT + ST + g) * WS + v, a.s.dec_proj + (size_t)slot * JOINT + c * KW + v);
                }
                cp_async16(st + (RT + g) * WS + v, src + v);
            }
        }
        cp_async_commit();                                                         // an empty group keeps the wait arithmetic uniform
    };

    for (int q = 0; q < NST - 1; ++q) issue(q);
    float tot[RPL][SPL];
    for (int q = 0; q < total_steps; ++q) {
        const int item = (int)blockIdx.x + (q / NCH) * (int)gridDim.x, c = q % NCH;
        const int rt = item % n_rt, s0 = (item / n_rt) * ST, ns = min(ST, n - s0);
        float* st = ring + (q % NST) * STAGE_F;
        cp_async_wait<NST - 2>();                                                 // this thread's copies of step q have landed
        if (MODE == MODE_JOINT) {                                                 // z = relu(enc_proj + pred_proj) once per element (nemo-ggml.cpp:1092-1094), by the thread that copied it
            for (int p = tid; p < ns * VPR; p += NT) {
                const int g = p / VPR, v = (p % VPR) * 4;
                float4 e = *reinterpret_cast<const float4*>(st + (RT + g) * WS + v);
                const float4 d = *reinterpret_cast<const float4*>(st + (RT + ST + g) * WS + v);
                e.x = fmaxf(e.x + d.x, 0.f); e.y = fmaxf(e.y + d.y, 0.f); e.z = fmaxf(e.z + d.z, 0.f); e.w = fmaxf(e.w + d.w, 0.f);
                *reinterpret_cast<float4*>(st + (RT + g) * WS + v) = e;
            }
        }
        __syncthreads();                                                          // step q visible to everyone; everyone is done with step q - 1
        issue(q + NST - 1);                                                       // refills the buffer step q - 1 used
        const float* wsm = st + (warp * 4 * RPL + rg * RPL) * WS;
        const float* xsm = st + (RT + sg) * WS;
        float acc[RPL][SPL];
#pragma unroll
        for (int i = 0; i < RPL; ++i)
#pragma unroll
            for (int j = 0; j < SPL; ++j) acc[i][j] = 0.f;
#pragma unroll 4
        for (int k = 0; k < KW; k += 4) {
            float4 w[RPL], x[SPL];
#pragma unroll
            for (int i = 0; i < RPL; ++i) w[i] = *reinterpret_cast<const float4*>(wsm + i * WS + k);
#pragma unroll
            for (int j = 0; j < SPL; ++j) x[j] = *reinterpret_cast<const float4*>(xsm + 8 * j * WS + k);
#pragma unroll
            for (int i = 0; i < RPL; ++i)
#pragma unroll
                for (int j = 0; j < SPL; ++j) {
                    acc[i][j] = fmaf(w[i].x, x[j].x, acc[i][j]); acc[i][j] = fmaf(w[i].y, x[j].y, acc[i][j]);
                    acc[i][j] = fmaf(w[i].z, x[j].z, acc[i][j]); acc[i][j] = fmaf(w[i].w, x[j].w, acc[i][j]);
                }
        }
#pragma unroll
        for (int i = 0; i < RPL; ++i)
#pragma unroll
            for (int j = 0; j < SPL; ++j) tot[i][j] = c == 0 ? acc[i][j] : tot[i][j] + acc[i][j];   // chunk order = phase()'s warp order
        if (c != NCH - 1) continue;
        // ---------------- the item is complete ----------------
        if (MODE == MODE_LSTM) {                                                  // gate order i,f,g,o (nemo-ggml.cpp:518-541)
#pragma unroll
            for (int i = 0; i < RPL; ++i)
#pragma unroll
                for (int j = 0; j < SPL; ++j) {
                    float gsum[4];
#pragma unroll
                    for (int qg = 0; qg < 4; ++qg) gsum[qg] = __shfl_sync(0xffffffffu, tot[i][j], qg * 8 + sg);
                    const int g = sg + 8 * j;
                    if (rg == (i & 3) && g < ns) {                                // one lane of the four finalises this (unit, stream)
                        const int b = sm.list[s0 + g], slot = sm.slot[b], par = sm.par[b];
                        const int u = rt * (8 * RPL) + warp * RPL + i;
                        float gate[4];
#pragma unroll
                        for (int qg = 0; qg < 4; ++qg) gate[qg] = (gsum[qg] + __ldg(a.w.b_ih[layer] + qg * HID + u)) + __ldg(a.w.b_hh[layer] + qg * HID + u);
                        const float ig = sigmoid_exact(gate[0]), fg = sigmoid_exact(gate[1]), gg = tanhf(gate[2]), og = sigmoid_exact(gate[3]);
                        const size_t o_old = (size_t)slot * 2 * PAR_STRIDE + par * PAR_STRIDE + layer * HID + u;
                        const size_t o_new = (size_t)slot * 2 * PAR_STRIDE + (par ^ 1) * PAR_STRIDE + layer * HID + u;
                        const float cn = fg * __ldcg(a.s.cbuf + o_old) + ig * gg;
                        a.s.cbuf[o_new] = cn; a.s.hbuf[o_new] = og * tanhf(cn);
                    }
                }
        } else if (MODE == MODE_PRED) {                                           // joint.pred (nemo-ggml.cpp:1086-1087)
#pragma unroll
            for (int i = 0; i < RPL; ++i)
#pragma unroll
                for (int j = 0; j < SPL; ++j) {
                    const int g = sg + 8 * j, row = rt * RT + warp * 4 * RPL + rg * RPL + i;
                    if (g < ns && row < JOINT) a.s.dec_proj[(size_t)sm.slot[sm.list[s0 + g]] * JOINT + row] = tot[i][j] + __ldg(a.w.pred_b + row);
                }
        } else {                                                                  // logits of this tile -> per-stream argmax key
#pragma unroll
            for (int j = 0; j < SPL; ++j) {
                const int g = sg + 8 * j;
                unsigned long long key = 0ull;
#pragma unroll
                for (int i = 0; i < RPL; ++i) {
                    const int v = rt * RT + warp * 4 * RPL + rg * RPL + i;
                    if (v < VOCAB && g < ns) {
                        const float sv = tot[i][j] + __ldg(a.w.out_b + v);
                        const unsigned long long kk = argmax_key(sv, v);             // largest logit, ties to the lowest index (:847-854)
                        key = kk > key ? kk : key;
                        if (a.logits_tap && sm.list[s0 + g] == 0 && ne0 < a.logits_tap_cap) a.logits_tap[(size_t)ne0 * VOCAB + v] = sv;
                    }
                }
                unsigned long long o = shfl_xor_u64(key, 8); key = o > key ? o : key;
                o = shfl_xor_u64(key, 16); key = o > key ? o : key;
                if (rg == 0) sm.keys[warp][g] = key;
            }
            __syncthreads();
            if (tid < ns) {
                unsigned long long key = sm.keys[0][tid];
#pragma unroll
                for (int w8 = 1; w8 < NW; ++w8) { const unsigned long long o = sm.keys[w8][tid]; key = o > key ? o : key; }
                atomicMax(a.best + (size_t)(round % 3) * a.B + sm.list[s0 + tid], key);
            }
            // sm.keys is rewritten at the end of the NEXT item at the earliest: at least one step barrier lies in between
        }
    }
    cp_async_wait<0>();
    __syncthreads();                                                              // the ring is free for whatever runs next
}


// ------------------------------------------------------------------------------------------
// phase_gemv(): the LSTM phase for a handful of streams (<= 8 SPL) on a NARROW grid (decode overlap: ~20 CTAs next to the next
// step's encoder). There a CTA owns 1/20 of the gate matrix and the phase is bound by how fast 256 threads can issue, so the tile is
// built around instructions per FMA: 128 weight rows = 32 hidden units x 4 gates per CTA tile, a lane owns ONE unit (all four gates:
// no shuffle, every thread finalises its own cell) x SPL streams = 4 + SPL shared-memory loads per 16 SPL FMAs (phase_pipe<1,1>: 2 per
// 4). K streams through a 4-stage cp.async ring in steps of 80; the 160-wide chunk partials are formed and added exactly as in
// phase() / phase_pipe(): same bits.
// Stage layout: weight row (gate g, unit index i) at row g * 32 + i, so the four units a warp's row groups read sit in different
// banks; stream vectors behind them.
// ------------------------------------------------------------------------------------------
template <int SPL>
__device__ void phase_gemv(const DecodeArgs& a, DecSmem& sm, int layer, int n) {
    constexpr int NSUB = 16, KS = 2 * HID / NSUB, WS = KS + 4, VPR = KS / 4;       // 16 pipeline steps of 80 floats = 8 chunks of 160
    constexpr int UT = 32, RT = 4 * UT, ST = 8 * SPL;
    constexpr int STAGE_F = (RT + ST) * WS;
    constexpr int NST = NW * STAGE_FLOATS / STAGE_F > 5 ? 5 : NW * STAGE_FLOATS / STAGE_F;
    static_assert(NST >= 3, "at least three stages in the ring");
    const int n_rt = HID / UT, n_sb = (n + ST - 1) / ST, n_items = n_rt * n_sb;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, rgrp = lane >> 3, sg = lane & 7;
    const int my_items = (int)blockIdx.x < n_items ? (n_items - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;
    const int total_steps = my_items * NSUB;
    float* ring = &sm.stage[0][0];

    auto issue = [&](int q) {
        if (q < total_steps) {
            const int item = (int)blockIdx.x + (q / NSUB) * (int)gridDim.x, sub = q % NSUB;
            const int rt = item % n_rt, s0 = (item / n_rt) * ST, ns = min(ST, n - s0);
            const bool rec = sub >= NSUB / 2;                                     // k >= 640: recurrent half
            const int kc = (sub % (NSUB / 2)) * KS;
            const float* wmat = rec ? a.w.w_hh[layer] : a.w.w_ih[layer];
            float* st = ring + (q % NST) * STAGE_F;
            for (int p = tid; p < RT * VPR; p += NT) {
                const int rr = p / VPR, v = (p % VPR) * 4;
                const int row = (rr / UT) * HID + rt * UT + (rr % UT);            // gate * 640 + unit
                cp_async16(st + rr * WS + v, wmat + (size_t)row * HID + kc + v);
            }
            for (int p = tid; p < ns * VPR; p += NT) {
                const int g = p / VPR, v = (p % VPR) * 4;
                const int b = sm.list[s0 + g], slot = sm.slot[b], par = sm.par[b];
                const float* hb = a.s.hbuf + (size_t)slot * 2 * PAR_STRIDE;
                const float* src = rec ? hb + par * PAR_STRIDE + layer * HID                                   // committed h of this layer
                                       : (layer == 0 ? a.w.embed + (size_t)sm.prev[b] * HID                    // nemo-stream.cpp:825-828
                                                     : hb + (par ^ 1) * PAR_STRIDE);                           // layer-1 input = layer-0 h'
                cp_async16(st + (RT + g) * WS + v, src + kc + v);
            }
        }
        cp_async_commit();
    };

    for (int q = 0; q < NST - 1; ++q) issue(q);
    float tot[4][SPL], acc[4][SPL];
    for (int q = 0; q < total_steps; ++q) {
        const int item = (int)blockIdx.x + (q / NSUB) * (int)gridDim.x, sub = q % NSUB;
        const int rt = item % n_rt, s0 = (item / n_rt) * ST, ns = min(ST, n - s0);
        const float* st = ring + (q % NST) * STAGE_F;
        cp_async_wait<NST - 2>();
        __syncthreads();
        issue(q + NST - 1);
        if ((sub & 1) == 0) {
#pragma unroll
            for (int g = 0; g < 4; ++g)
#pragma unroll
                for (int j = 0; j < SPL; ++j) acc[g][j] = 0.f;
        }
        const float* wsm = st + (warp * 4 + rgrp) * WS;
        const float* xsm = st + (RT + sg) * WS;
#pragma unroll 5
        for (int k = 0; k < KS; k += 4) {
            float4 w[4], x[SPL];
#pragma unroll
            for (int g = 0; g < 4; ++g) w[g] = *reinterpret_cast<const float4*>(wsm + g * UT * WS + k);
#pragma unroll
            for (int j = 0; j < SPL; ++j) x[j] = *reinterpret_cast<const float4*>(xsm + 8 * j * WS + k);
#pragma unroll
            for (int g = 0; g < 4; ++g)
#pragma unroll
                for (int j = 0; j < SPL; ++j) {
                    acc[g][j] = fmaf(w[g].x, x[j].x, acc[g][j]); acc[g][j] = fmaf(w[g].y, x[j].y, acc[g][j]);
                    acc[g][j] = fmaf(w[g].z, x[j].z, acc[g][j]); acc[g][j] = fmaf(w[g].w, x[j].w, acc[g][j]);
                }
        }
        if ((sub & 1) == 0) continue;                                             // second half of a 160-wide chunk: its partial is complete
#pragma unroll
        for (int g = 0; g < 4; ++g)
#pragma unroll
            for (int j = 0; j < SPL; ++j) tot[g][j] = sub == 1 ? acc[g][j] : tot[g][j] + acc[g][j];
        if (sub != NSUB - 1) continue;
        // ---------------- the unit's four gate sums are complete, in this lane: cell update (nemo-ggml.cpp:518-541) ----------------
#pragma unroll
        for (int j = 0; j < SPL; ++j) {
            const int g = sg + 8 * j;
            if (g >= ns) continue;
            const int b = sm.list[s0 + g], slot = sm.slot[b], par = sm.par[b];
            const int u = rt * UT + warp * 4 + rgrp;
            float gate[4];
#pragma unroll
            for (int qg = 0; qg < 4; ++qg) gate[qg] = (tot[qg][j] + __ldg(a.w.b_ih[layer] + qg * HID + u)) + __ldg(a.w.b_hh[layer] + qg * HID + u);
            const float ig = sigmoid_exact(gate[0]), fg = sigmoid_exact(gate[1]), gg = tanhf(gate[2]), og = sigmoid_exact(gate[3]);
            const size_t o_old = (size_t)slot * 2 * PAR_STRIDE + par * PAR_STRIDE + layer * HID + u;
            const size_t o_new = (size_t)slot * 2 * PAR_STRIDE + (par ^ 1) * PAR_STRIDE + layer * HID + u;
            const float cn = fg * __ldcg(a.s.cbuf + o_old) + ig * gg;
            a.s.cbuf[o_new] = cn; a.s.hbuf[o_new] = og * tanhf(cn);
        }
    }
    cp_async_wait<0>();
    __syncthreads();
}

template <int MODE>
__device__ __forceinline__ void phase_dispatch(const DecodeArgs& a, DecSmem& sm, int layer, int n, int round, int ne0) {
    // one or two items per CTA and phase (full-width grid, a handful of streams): the one-shot staging of phase(); a narrow grid (decode
    // overlap) or many stream blocks: the pipelined tiles. Same arithmetic, same bits (see phase_pipe).
    const bool narrow = gridDim.x <= 64;
    const bool pipe = narrow || n >= a.pipe_min_n;
    constexpr int RPL = MODE == MODE_LSTM ? 5 : 2;
    if (!pipe) {
        if (n <= 8) phase<RPL, 1, MODE>(a, sm, layer, n, round, ne0);
        else phase<RPL, 2, MODE>(a, sm, layer, n, round, ne0);
        return;
    }
    if (narrow && MODE == MODE_LSTM && n <= 16) {                                 // few emitting streams on a narrow grid: one unit per lane
        if (n <= 8) phase_gemv<1>(a, sm, layer, n); else phase_gemv<2>(a, sm, layer, n);
        return;
    }
    if (narrow && MODE == MODE_JOINT && n > 16) { phase_pipe<2, 4, MODE>(a, sm, layer, n, round, ne0); return; }   // fewer instructions per FMA than <1,4>
    if (n <= 8) phase_pipe<1, 1, MODE>(a, sm, layer, n, round, ne0);
    else if (n <= 16) phase_pipe<1, 2, MODE>(a, sm, layer, n, round, ne0);
    else if (n <= 64) phase_pipe<1, 4, MODE>(a, sm, layer, n, round, ne0);        // more (smaller) tiles while the stream blocks are few
    else phase_pipe<2, 4, MODE>(a, sm, layer, n, round, ne0);
}

__global__ void __launch_bounds__(NT, 1) rnnt_decode_kernel(const DecodeArgs a) {
    extern __shared__ __align__(16) uint8_t dec_smem_raw[];
    DecSmem& sm = *reinterpret_cast<DecSmem*>(dec_smem_raw);
    const int tid = threadIdx.x, B = a.B, T = a.T;
    const unsigned nblk = gridDim.x;
    unsigned epoch = 0;
    int tr_slot = -1;
    if (trace_thread()) { tr_slot = trace_begin(TR_DECODE); trace_mark(tr_slot, 1); }
    int ne0 = 0;                                                                  // joint evaluations of batch row 0 so far (debug tap)

    for (int b = tid; b < B; b += NT) {
        const int slot = a.slot_of_b[b];
        sm.slot[b] = slot; sm.prev[b] = a.s.prev_token[slot]; sm.par[b] = (unsigned char)(a.s.par[slot] & 1);
        sm.need[b] = a.s.cand_valid[slot] ? 0 : 1;
        sm.fi[b] = 0; sm.oc[b] = 0; sm.sc[b] = 0;
    }
    __syncthreads();

    // trace (block 0 only): t[3] = ns spent in prediction-network phases (incl. their 3 grid barriers), t[4] = ns in joint + argmax
    // phases, t[5] = rounds << 32 | rounds that ran the prediction network
    unsigned long long tr_pred = 0, tr_joint = 0, tr_rounds = 0, tr_t = 0;
    for (int round = 0;; ++round) {
        // ---------------- prediction network for active streams whose candidate is stale ----------------
        const int n_need = compact(sm, B, [&](int b) { return sm.need[b] != 0 && sm.fi[b] < T; });
        if (tr_slot >= 0) tr_t = gtime();
        if (n_need > 0) {
            phase_dispatch<MODE_LSTM>(a, sm, 0, n_need, round, ne0);
            grid_barrier(a.barrier, epoch, nblk);
            phase_dispatch<MODE_LSTM>(a, sm, 1, n_need, round, ne0);
            grid_barrier(a.barrier, epoch, nblk);
            phase_dispatch<MODE_PRED>(a, sm, 0, n_need, round, ne0);
            grid_barrier(a.barrier, epoch, nblk);
            for (int i = tid; i < n_need; i += NT) sm.need[sm.list[i]] = 0;
            __syncthreads();
            if (tr_slot >= 0) { const unsigned long long t1 = gtime(); tr_pred += t1 - tr_t; tr_t = t1; tr_rounds += 1; }
        }
        // ---------------- joint + argmax ----------------
        const int n_act = compact(sm, B, [&](int b) { return sm.fi[b] < T; });
        if (n_act == 0) break;                                                    // identical in every CTA
        phase_dispatch<MODE_JOINT>(a, sm, 0, n_act, round, ne0);
        grid_barrier(a.barrier, epoch, nblk);
        if (blockIdx.x == 0)                                                      // keys of round+2: everyone is done reading them (see header)
            for (int b = tid; b < B; b += NT) a.best[(size_t)((round + 2) % 3) * B + b] = 0ull;
        // ---------------- decision, replicated in every CTA (:856-874) ----------------
        for (int i = tid; i < n_act; i += NT) {
            const int b = sm.list[i];
            const unsigned long long key = __ldcg(a.best + (size_t)(round % 3) * B + b);
            const int tok = (int)(0xFFFFFFFFu - (unsigned)(key & 0xFFFFFFFFull));
            if (tok == BLANK) { sm.fi[b] += 1; sm.sc[b] = 0; }                    // blank: next frame, state untouched
            else {
                if (blockIdx.x == 0) {
                    a.out_tokens[(size_t)b * MAX_SYMBOLS * T + sm.oc[b]] = tok;
                    if (a.out_frames) a.out_frames[(size_t)b * MAX_SYMBOLS * T + sm.oc[b]] = sm.fi[b];   // nemo-ggml.cpp:1240 tokens.push_back({best_token, t})
                }
                sm.oc[b] += 1; sm.prev[b] = tok; sm.par[b] ^= 1; sm.need[b] = 1;  // emit: commit the candidate (parity flip)
                if (sm.sc[b] + 1 >= MAX_SYMBOLS) { sm.fi[b] += 1; sm.sc[b] = 0; } else sm.sc[b] += 1;   // :813
            }
        }
        if (sm.list[0] == 0) ne0 += 1;                                            // list is ascending: row 0 is first whenever it was evaluated
        __syncthreads();                                                          // state updates visible before the next compaction
        if (tr_slot >= 0) { tr_joint += gtime() - tr_t; tr_rounds += 1ull << 32; }
    }
    if (blockIdx.x == 0) {
        for (int b = tid; b < B; b += NT) {
            const int slot = sm.slot[b];
            a.s.prev_token[slot] = sm.prev[b]; a.s.par[slot] = sm.par[b]; a.s.cand_valid[slot] = sm.need[b] ? 0 : 1;
            a.out_count[b] = sm.oc[b];
        }
        if (tid == 0 && a.logits_tap_n) *a.logits_tap_n = ne0;
        if (tid == 0 && tr_slot >= 0) {
            trace_mark(tr_slot, 2);
            c_trace->rec[tr_slot].t[3] = tr_pred; c_trace->rec[tr_slot].t[4] = tr_joint; c_trace->rec[tr_slot].t[5] = tr_rounds;
        }
    }
}
}  // namespace

static int decode_grid() {                 // per device ordinal: the attribute below and the SM count belong to the CURRENT device
    static std::atomic<int> grids[MAX_DEVICES];
    int dev = 0;
    NSB_CUDA(cudaGetDevice(&dev));
    std::atomic<int>& g = grids[dev & (MAX_DEVICES - 1)];
    if (g.load(std::memory_order_acquire) == 0) {
        int sms = 0, per_sm = 0;
        NSB_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
        NSB_CUDA(cudaFuncSetAttribute(rnnt_decode_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(DecSmem)));
        NSB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, rnnt_decode_kernel, NT, sizeof(DecSmem)));
        if (per_sm < 1) throw CudaError("decode kernel cannot be resident");
        g.store(sms, std::memory_order_release);                                  // one CTA per SM: co-residency guaranteed
    }
    return g.load(std::memory_order_acquire);
}
size_t decode_sync_bytes(int B) { return 16 + (size_t)3 * B * sizeof(unsigned long long); }

int decode_narrow_ctas() {
    static const int n = [] { const char* e = getenv("NSB_DECODE_CTAS"); const int v = e ? atoi(e) : 20; return std::max(2, v & ~1); }();
    return n;
}

// narrow_ctas = 0: one CTA per SM, cooperative launch (the decode has the GPU to itself). narrow_ctas > 0: that many CTAs, launched as
// CTA pairs (clusters of 2: a pair takes one TPC, so the CTA-pair GEMMs of a concurrently running encoder keep their TPCs whole) with a
// plain launch: the kernel then shares the GPU with the next step's encoder. Its grid barrier needs every CTA resident at some
// point, which a grid this small reaches as soon as a few SMs are free -- nothing the other kernels run ever waits on this one.
int launch_decode(const DecodeArgs& a_in, void* sync_buf, cudaStream_t st, int narrow_ctas, int pipe_min_n) {
    const int full = decode_grid();
    if (a_in.B > MAXB) throw CudaError("decode: more than 1024 streams in one step");
    DecodeArgs a = a_in;
    // full-width grid: pipelined tiles from this many streams per phase on (below, one or two one-shot items per CTA are as good or better)
    static const int pipe_n = [] { const char* e = getenv("NSB_DECODE_PIPE_N"); return e ? atoi(e) : 65; }();
    a.pipe_min_n = pipe_min_n > 0 ? pipe_min_n : pipe_n;
    a.barrier = reinterpret_cast<unsigned*>(sync_buf);
    a.best = reinterpret_cast<unsigned long long*>((char*)sync_buf + 16);
    NSB_CUDA(cudaMemsetAsync(sync_buf, 0, decode_sync_bytes(a.B), st));           // barrier counter + argmax keys
    if (narrow_ctas > 0 && narrow_ctas < full) {
        cudaLaunchConfig_t cfg{};
        cfg.gridDim = dim3(narrow_ctas); cfg.blockDim = dim3(NT); cfg.dynamicSmemBytes = sizeof(DecSmem); cfg.stream = st;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeClusterDimension; at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
        cfg.attrs = at; cfg.numAttrs = 1;
        NSB_CUDA(cudaLaunchKernelEx(&cfg, rnnt_decode_kernel, a));
        return narrow_ctas;
    }
    void* args[] = {(void*)&a};
    NSB_CUDA(cudaLaunchCooperativeKernel((void*)rnnt_decode_kernel, dim3(full), dim3(NT), args, sizeof(DecSmem), st));
    return full;
}

}  // namespace nsb
