// encoder.cu -- stage E: BERT / RoBERTa post-LN encoder forward -> unit-norm CLS rows.
//
// Replaces `self.model(**inputs).last_hidden_state[:, 0, :]` + F.normalize at
// /root/reference/src/adaptive_classifier/classifier.py:1271-1275 (HF BertModel.forward:
// embeddings modeling_bert.py:53-113, self-attention :143-207, output+LN :287-298, FFN :330-356).
//
// Precision: every tensor-core operand is fp16 (RNE from fp32), accumulation fp32 in TMEM, residual stream, LayerNorm,
// softmax and GELU in fp32.  fp16 carries the same 10-bit mantissa as tf32, so the measured error is the tf32 one
// (oracle/precision_study.py: 1.7e-4 on squared-L2 distances, bf16 would be 1.4e-3 > the 1e-3 tolerance) at twice the
// tensor rate and half the operand bytes.
//
//   projections   tcgen05 GEMM of gemm_tc.cuh (kind::f16) with compile-time-specialised fused epilogues:
//                 bias | bias+GELU(erf) | bias+residual, fp16 or fp32 output, V written TRANSPOSED per (sequence, head)
//   attention     one CTA per (sequence, head): Q, K and V^T tiles by TMA, QK^T and PV as tcgen05 MMAs with the score
//                 tile / output tile in TMEM, thread-per-query-row softmax in between (S <= 128, head_dim 64)
//   LayerNorm     never materialised inside the layer stack: the residual epilogues keep the un-normalised sums y (fp32) and
//                 per-row (sum, sumsq) partials, the consuming projections run on gamma-scaled weights and apply the
//                 rank-1 correction r (acc - mu c1) + c0 in their epilogue ("deferred LayerNorm" below)
#include "gemm_tc2.cuh"
#include <cuda_fp16.h>
#include <math_constants.h>
#include <vector>

namespace ac {

__device__ __forceinline__ float ex2_approx(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float rcp_approx(float x) {
    float y;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
// exact-erf GELU y*Phi(y) with erfc from Abramowitz-Stegun 7.1.26 (|error| < 1.5e-7 + 2 ulp of the two MUFU
// approximations).  With x = |y|/sqrt2, h = erfc(x)/2 = (poly(t)/2) * t * exp(-x^2), t = 1/(1 + p x):
//     y >= 0: y*(1 - h) = y - y*h        y < 0: y*h            =>   gelu(y) = max(y, 0) - |y*h|
// 2 MUFU + 12 FP32 ops per element and no branch/select.  The GELU epilogue touches 201 M elements per layer; the
// issue budget that hides it behind a K = 768 fp16 mainloop is ~24 instructions per element (libdevice erff alone ~30).
__device__ __forceinline__ float gelu_erf(float y) {
    const float ay = fabsf(y);
    const float t = rcp_approx(fmaf(0.3275911f * 0.70710678118654752440f, ay, 1.f));
    float p = fmaf(0.5f * 1.061405429f, t, 0.5f * -1.453152027f);
    p = fmaf(p, t, 0.5f * 1.421413741f);
    p = fmaf(p, t, 0.5f * -0.284496736f);
    p = fmaf(p, t, 0.5f * 0.254829592f);
    const float e = ex2_approx((y * y) * (-0.5f * 1.4426950408889634f));   // exp(-y^2/2)
    const float h = (p * t) * e;                                             // erfc(|y|/sqrt2) / 2
    return fmaxf(y, 0.f) - fabsf(y * h);
}

// ------------------------------------------------------------------------------------------------
// fused epilogue of the encoder linears (compile-time specialised)
//   MODE 0 bias, 1 bias + exact-erf GELU, 2 bias + fp32 residual;  OUT_HALF: fp16 output (next GEMM operand) or fp32
//   VT: columns >= vt_col0 (the V third of the fused QKV projection) are written transposed to
//       vT[(b*H + feature) * S_pad + key] so that attention can TMA-load V^T as a K-major B operand.
// ------------------------------------------------------------------------------------------------
//   DEFER: the A operand was the UN-normalised residual sum y (fp16) and the weights were packed as fp16(gamma * W):
//       LayerNorm(y) W^T + b = r (acc - mu c1) + c0  with the row statistics (mu, r) of y, c1 = rowsum(W'), and
//       `bias` holding c0 = W beta + b  (see "deferred LayerNorm" below)
//   COLS:  accumulator columns one epilogue warp drains per tile (128 with 8 epilogue warps, 64 with 16): only the DEFER
//          variant needs it, to know which chunk is the first of its slice
template <int MODE, bool OUT_HALF, bool VT, bool DEFER = false, int COLS = GEMM_BLOCK_N / 2>
struct EpiLinear {
    static_assert(!DEFER || (OUT_HALF && MODE != 2), "the deferred-LayerNorm consumer epilogues write fp16 operands");
    const float *__restrict__ bias;       // [N]   (DEFER: c0)
    const float *__restrict__ residual;   // [M, ldy] (MODE 2)
    void *Y;                              // [M, ldy] fp16 or fp32
    int M, N, ldy;
    int round_out;                        // fp32 output only: round to tf32 (tests of the tf32 path)
    __half *vT;                           // VT only
    int vt_col0, S, S_pad, H;
    const float *__restrict__ c1;         // DEFER only: [N] row sums of the packed weight
    const float2 *__restrict__ row_stats; // DEFER only: [M] (mu, 1/sqrt(var + eps)) of the A rows

    static constexpr int kUnrollChunks = 4;   // `buf` must be a compile-time constant (register double buffer)
    static constexpr int kPrefetchDist = 1;
    struct State {
        // residual (MODE 2) of one 32-column chunk in the layout of the transposed phase: [column half][row pass],
        // double-buffered so chunk c+1 is in flight while chunk c is processed
        float4 res[(MODE == 2) ? 2 : 1][(MODE == 2) ? 8 : 1];
        float mu, r;                      // DEFER: statistics of this thread's accumulator row
    };
    // accumulator + bias, or the deferred-LayerNorm form r (acc - mu c1) + c0
    __device__ __forceinline__ float pre(const State &st, float acc, float b, float c1v) const {
        return DEFER ? fmaf(st.r, fmaf(-st.mu, c1v, acc), b) : acc + b;
    }
    __device__ __forceinline__ void begin_cta(State &, int, int) const {}
    __device__ __forceinline__ void end_cta(State &, int, int) const {}

    __device__ __forceinline__ float act(float y) const {
        if (MODE == 1) y = gelu_erf(y);
        return y;
    }

    // transposed phase mapping (fp32 staging holds 16 columns at a time): lane = (r8 = lane / 4, c = lane % 4) handles
    // rows r8 + 8*i (i < 4) and the 16-byte column group c of each 16-column half.
    __device__ __forceinline__ void prefetch(State &st, const GemmTileInfo &ti, int row, int col0, int lane, int buf) const {
        if (DEFER) {
            if (((col0 - ti.n0) & (COLS - 1)) == 0) {                  // first chunk of this warp's column slice
                const float2 ms = (row < M) ? __ldg(row_stats + row) : make_float2(0.f, 0.f);
                st.mu = ms.x;
                st.r = ms.y;
            }
        }
        if (MODE != 2) return;
        const int row_base = ti.m0 + ((threadIdx.x >> 5) & 3) * 32;
        const int r8 = lane >> 2, c = lane & 3;
#pragma unroll
        for (int half = 0; half < 2; ++half) {
            const int col = col0 + 16 * half + 4 * c;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int grow = row_base + r8 + 8 * i;
                st.res[buf][half * 4 + i] =
                    (grow < M && col + 4 <= N)
                        ? __ldg(reinterpret_cast<const float4 *>(residual + static_cast<int64_t>(grow) * ldy + col))
                        : make_float4(0, 0, 0, 0);
            }
        }
    }

    __device__ __forceinline__ void tile(State &st, const GemmTileInfo &ti, int row, int col0, const float (&v)[32],
                                         uint8_t *stage, int lane, int buf, uint32_t /*taddr*/) const {
        const int row_base = ti.m0 + ((threadIdx.x >> 5) & 3) * 32;        // first row of this warp's TMEM quarter
        if (row_base >= M || col0 >= N) return;                              // warp-uniform
        if (VT && col0 >= vt_col0) {
            // thread = token row: lanes hold 32 consecutive keys of (mostly) one sequence -> 64-byte coalesced stores
            if (row < M) {
                const int b = row / S, key = row - b * S;
                __half *dst = vT + (static_cast<int64_t>(b) * H + (col0 - vt_col0)) * S_pad + key;
#pragma unroll
                for (int j = 0; j < 32; j += 4) {
                    const float4 b4 = __ldg(reinterpret_cast<const float4 *>(bias + col0 + j));
                    const float4 c4 = DEFER ? __ldg(reinterpret_cast<const float4 *>(c1 + col0 + j)) : make_float4(0, 0, 0, 0);
                    dst[static_cast<int64_t>(j) * S_pad] = __float2half_rn(pre(st, v[j], b4.x, c4.x));
                    dst[static_cast<int64_t>(j + 1) * S_pad] = __float2half_rn(pre(st, v[j + 1], b4.y, c4.y));
                    dst[static_cast<int64_t>(j + 2) * S_pad] = __float2half_rn(pre(st, v[j + 2], b4.z, c4.z));
                    dst[static_cast<int64_t>(j + 3) * S_pad] = __float2half_rn(pre(st, v[j + 3], b4.w, c4.w));
                }
            }
            return;
        }
        if (OUT_HALF) {
            // stage 32 rows x 32 halves (64 B payload per 80-byte row), then lane (r4 = lane/4 .. 8 rows per pass, c8 = lane%4)
            uint4 *srow = reinterpret_cast<uint4 *>(stage + lane * GEMM_EPI_STAGE_ROW_BYTES);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float4 ba = __ldg(reinterpret_cast<const float4 *>(bias + col0 + 8 * j));
                const float4 bb = __ldg(reinterpret_cast<const float4 *>(bias + col0 + 8 * j + 4));
                const float4 ca = DEFER ? __ldg(reinterpret_cast<const float4 *>(c1 + col0 + 8 * j)) : make_float4(0, 0, 0, 0);
                const float4 cb = DEFER ? __ldg(reinterpret_cast<const float4 *>(c1 + col0 + 8 * j + 4)) : make_float4(0, 0, 0, 0);
                float y[8];
                y[0] = act(pre(st, v[8 * j], ba.x, ca.x)); y[1] = act(pre(st, v[8 * j + 1], ba.y, ca.y));
                y[2] = act(pre(st, v[8 * j + 2], ba.z, ca.z)); y[3] = act(pre(st, v[8 * j + 3], ba.w, ca.w));
                y[4] = act(pre(st, v[8 * j + 4], bb.x, cb.x)); y[5] = act(pre(st, v[8 * j + 5], bb.y, cb.y));
                y[6] = act(pre(st, v[8 * j + 6], bb.z, cb.z)); y[7] = act(pre(st, v[8 * j + 7], bb.w, cb.w));
                uint4 pk;
                __half2 h0 = __floats2half2_rn(y[0], y[1]), h1 = __floats2half2_rn(y[2], y[3]);
                __half2 h2 = __floats2half2_rn(y[4], y[5]), h3 = __floats2half2_rn(y[6], y[7]);
                pk.x = *reinterpret_cast<uint32_t *>(&h0); pk.y = *reinterpret_cast<uint32_t *>(&h1);
                pk.z = *reinterpret_cast<uint32_t *>(&h2); pk.w = *reinterpret_cast<uint32_t *>(&h3);
                srow[j] = pk;
            }
            __syncwarp();
            const int r8 = lane >> 2, c = lane & 3;                           // 8 rows x 4 x 16 B per pass
            __half *Yh = static_cast<__half *>(Y);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int rr = r8 + 8 * i;
                const int grow = row_base + rr;
                const int col = col0 + 8 * c;
                if (grow < M && col + 8 <= N) {
                    const uint4 pk = *reinterpret_cast<const uint4 *>(stage + rr * GEMM_EPI_STAGE_ROW_BYTES + 16 * c);
                    *reinterpret_cast<uint4 *>(Yh + static_cast<int64_t>(grow) * ldy + col) = pk;
                }
            }
            __syncwarp();
        } else {
            // fp32 output (pre-LayerNorm sums): two passes of 16 columns through the staging tile
            float *Yf = static_cast<float *>(Y);
            const int r8 = lane >> 2, c = lane & 3;
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                const int col = col0 + 16 * half + 4 * c;
                float4 *srow = reinterpret_cast<float4 *>(stage + lane * GEMM_EPI_STAGE_ROW_BYTES);
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    srow[j] = make_float4(v[16 * half + 4 * j], v[16 * half + 4 * j + 1], v[16 * half + 4 * j + 2],
                                          v[16 * half + 4 * j + 3]);
                __syncwarp();
                const float4 b4 = (col + 4 <= N) ? __ldg(reinterpret_cast<const float4 *>(bias + col)) : make_float4(0, 0, 0, 0);
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const int rr = r8 + 8 * i;
                    const int grow = row_base + rr;
                    if (grow < M && col + 4 <= N) {
                        const float4 a = *reinterpret_cast<const float4 *>(stage + rr * GEMM_EPI_STAGE_ROW_BYTES + 16 * c);
                        float4 o;
                        o.x = act(a.x + b4.x); o.y = act(a.y + b4.y); o.z = act(a.z + b4.z); o.w = act(a.w + b4.w);
                        if (MODE == 2) {
                            const float4 rs = st.res[buf][half * 4 + i];    // requested one chunk ago
                            o.x += rs.x; o.y += rs.y; o.z += rs.z; o.w += rs.w;
                        }
                        if (round_out) { o.x = round_tf32(o.x); o.y = round_tf32(o.y); o.z = round_tf32(o.z); o.w = round_tf32(o.w); }
                        *reinterpret_cast<float4 *>(Yf + static_cast<int64_t>(grow) * ldy + col) = o;
                    }
                }
                __syncwarp();
            }
        }
    }
};

// ------------------------------------------------------------------------------------------------
// deferred LayerNorm: residual epilogue that never materialises LayerNorm
//
//   y_new = acc + bias + LN_prev(y_old)          LN_prev(y) = (y - mu) r gamma + beta recomputed from the fp32 y_old, its
//                                                row statistics and the pending LayerNorm's parameters
//   writes y_new (fp32, IN PLACE over y_old: every element is read and written by the same thread), fp16(y_new) (the
//   next GEMM's A operand, consumed through EpiLinear<.., DEFER = true>) and per-row partial (sum, sum of squares) of
//   this warp's 128 columns into parts[column part][row]; ln_stats_kernel turns the parts into (mu, r).
//   HBM traffic per half layer at B*S = 65536, H = 768: read y 201 MB, write y 201 MB + fp16 101 MB = 503 MB instead of
//   905 MB (GEMM epilogue 402 MB + LayerNorm kernel 503 MB); precision: oracle/deferred_ln_study.py (CPU emulation) and tests/test_gpu_parity.py (non-trivial gamma / beta).
// ------------------------------------------------------------------------------------------------
struct EpiResidDefer {
    const float *__restrict__ bias;        // [N]
    float *y;                              // [M, ld] fp32 residual sums: read (old) and written (new) in place
    __half *yh;                            // [M, ld] fp16 copy of the new sums
    const float2 *__restrict__ stats_prev; // [M] (mu, r) of the old sums
    const float *__restrict__ gamma;       // [N] pending LayerNorm of the old sums
    const float *__restrict__ beta;        // [N]
    float2 *parts;                         // [N / 128][part_stride] partial (sum, sumsq) of the new sums
    int64_t part_stride;
    int M, N, ld;

    static constexpr int kUnrollChunks = 4;
    // The residual epilogues move 327 KB per 128 x 256 tile (fp32 sums read + written, fp16 copy written) against a 3-13 us
    // mainloop: they are HBM-bound, and with one 4 KB chunk per warp in flight the 8 epilogue warps of an SM sustain ~25 GB/s
    // (3.65 TB/s over the chip; out-proj 152 us against an 85 us traffic floor).  Requesting two chunks ahead needs a third
    // 32-register buffer: with the 168 registers a 10-warp CTA can have (warps are allocated in fours) it spills, and measured
    // SLOWER on a B200 (14.5-14.8 ms per step against 13.9-14.1: profiles/r02_variants.md), so the distance stays 1.
    // Asking L2 for the next tile's rows one tile ahead (prefetch.global.L2, no registers) was also measured: 14.07 ms (one
    // request per 128 bytes) and 14.21 ms (per 32-byte sector) against 13.90-13.94 ms without, same box, same run -- the step
    // runs against the board's power cap (SM clock 1.5-1.7 GHz of 1.965), and extra requests in flight cost more clock than the
    // shorter load latency returns.
#ifndef AC_RESID_PREFETCH
#define AC_RESID_PREFETCH 1
#endif
    static constexpr int kPrefetchDist = AC_RESID_PREFETCH;
    struct State {
        float4 res[kPrefetchDist + 1][8];  // old sums of 32-column chunks (transposed-phase layout), one buffer more than the distance
        float2 ms[4];                      // (mu, r) of this lane's 4 rows (r8 + 8 i)
        float sum[4], sq[4];               // running partials of the new sums over this warp's 128 columns
    };
    __device__ __forceinline__ void begin_cta(State &, int, int) const {}
    __device__ __forceinline__ void end_cta(State &, int, int) const {}

    __device__ __forceinline__ void prefetch(State &st, const GemmTileInfo &ti, int, int col0, int lane, int buf) const {
        const int row_base = ti.m0 + ((threadIdx.x >> 5) & 3) * 32;
        const int r8 = lane >> 2, c = lane & 3;
        if (((col0 - ti.n0) & (GEMM_BLOCK_N / 2 - 1)) == 0) {           // first chunk of this warp's column half
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int grow = row_base + r8 + 8 * i;
                st.ms[i] = (grow < M) ? __ldg(stats_prev + grow) : make_float2(0.f, 0.f);
                st.sum[i] = 0.f;
                st.sq[i] = 0.f;
            }
        }
#pragma unroll
        for (int half = 0; half < 2; ++half) {
            const int col = col0 + 16 * half + 4 * c;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int grow = row_base + r8 + 8 * i;
                // plain (coherent) load: y is written by this very kernel, although never the element being read here
                st.res[buf][half * 4 + i] = (grow < M && col + 4 <= N)
                                                ? *reinterpret_cast<const float4 *>(y + static_cast<int64_t>(grow) * ld + col)
                                                : make_float4(0, 0, 0, 0);
            }
        }
    }

    __device__ __forceinline__ void tile(State &st, const GemmTileInfo &ti, int, int col0, const float (&v)[32], uint8_t *stage,
                                         int lane, int buf, uint32_t) const {
        const int row_base = ti.m0 + ((threadIdx.x >> 5) & 3) * 32;
        if (row_base >= M || col0 >= N) return;                              // warp-uniform
        const int r8 = lane >> 2, c = lane & 3;
#pragma unroll
        for (int half = 0; half < 2; ++half) {
            const int col = col0 + 16 * half + 4 * c;
            float4 *srow = reinterpret_cast<float4 *>(stage + lane * GEMM_EPI_STAGE_ROW_BYTES);
#pragma unroll
            for (int j = 0; j < 4; ++j)
                srow[j] = make_float4(v[16 * half + 4 * j], v[16 * half + 4 * j + 1], v[16 * half + 4 * j + 2], v[16 * half + 4 * j + 3]);
            __syncwarp();
            const bool col_ok = col + 4 <= N;
            const float4 b4 = col_ok ? __ldg(reinterpret_cast<const float4 *>(bias + col)) : make_float4(0, 0, 0, 0);
            const float4 g4 = col_ok ? __ldg(reinterpret_cast<const float4 *>(gamma + col)) : make_float4(0, 0, 0, 0);
            const float4 e4 = col_ok ? __ldg(reinterpret_cast<const float4 *>(beta + col)) : make_float4(0, 0, 0, 0);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int rr = r8 + 8 * i;
                const int grow = row_base + rr;
                if (grow < M && col_ok) {
                    const float4 a = *reinterpret_cast<const float4 *>(stage + rr * GEMM_EPI_STAGE_ROW_BYTES + 16 * c);
                    const float4 rs = st.res[buf][half * 4 + i];             // old sums, requested one chunk ago
                    const float mu = st.ms[i].x, r = st.ms[i].y;
                    float4 o;
                    o.x = (a.x + b4.x) + fmaf((rs.x - mu) * r, g4.x, e4.x);
                    o.y = (a.y + b4.y) + fmaf((rs.y - mu) * r, g4.y, e4.y);
                    o.z = (a.z + b4.z) + fmaf((rs.z - mu) * r, g4.z, e4.z);
                    o.w = (a.w + b4.w) + fmaf((rs.w - mu) * r, g4.w, e4.w);
                    *reinterpret_cast<float4 *>(y + static_cast<int64_t>(grow) * ld + col) = o;
                    const __half2 h0 = __floats2half2_rn(o.x, o.y), h1 = __floats2half2_rn(o.z, o.w);
                    uint2 pk;
                    pk.x = *reinterpret_cast<const uint32_t *>(&h0);
                    pk.y = *reinterpret_cast<const uint32_t *>(&h1);
                    *reinterpret_cast<uint2 *>(yh + static_cast<int64_t>(grow) * ld + col) = pk;
                    st.sum[i] += (o.x + o.y) + (o.z + o.w);
                    st.sq[i] += (o.x * o.x + o.y * o.y) + (o.z * o.z + o.w * o.w);
                }
            }
            __syncwarp();
        }
        if (((col0 - ti.n0) & (GEMM_BLOCK_N / 2 - 1)) == GEMM_BLOCK_N / 2 - 32) {   // last chunk of this warp's column half
            const int part = col0 / (GEMM_BLOCK_N / 2);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                float s = st.sum[i], q = st.sq[i];
                s += __shfl_xor_sync(0xffffffffu, s, 1);
                q += __shfl_xor_sync(0xffffffffu, q, 1);
                s += __shfl_xor_sync(0xffffffffu, s, 2);
                q += __shfl_xor_sync(0xffffffffu, q, 2);
                const int grow = row_base + r8 + 8 * i;
                if (c == 0 && grow < M) parts[static_cast<int64_t>(part) * part_stride + grow] = make_float2(s, q);
            }
        }
    }
};

// (sum, sumsq) partials of every 128-column part -> (mu, 1/sqrt(var + eps)) per row; parts are added in a fixed order.
// Kept as a kernel of its own (24 launches of ~3 us per forward): folding these six loads + rsqrt into the consuming epilogues
// was measured on a B200 and LOST 1 ms per step (35.5 k instead of 37.7 k queries/s, profiles/r02_bench_lnstats_folded.json):
// the loads sit at the head of every tile's epilogue, which is the critical path of the HBM-bound residual GEMMs.
__global__ void ln_stats_kernel(const float2 *__restrict__ parts, int nparts, int64_t part_stride, int rows, int H, float eps,
                                float2 *__restrict__ stats) {
    const int row = blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= rows) return;
    float s = 0.f, q = 0.f;
    for (int p = 0; p < nparts; ++p) {
        const float2 v = parts[static_cast<int64_t>(p) * part_stride + row];
        s += v.x;
        q += v.y;
    }
    const float mu = s / static_cast<float>(H);
    const float var = fmaxf(q / static_cast<float>(H) - mu * mu, 0.f);
    stats[row] = make_float2(mu, 1.f / sqrtf(var + eps));
}

__global__ void fill_stats_identity_kernel(float2 *__restrict__ stats, int64_t n) {
    const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i < n) stats[i] = make_float2(0.f, 1.f);
}
__global__ void fill_value_kernel(float *__restrict__ p, int n, float v) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}

// weight packing of a deferred-LayerNorm consumer (one warp per output row n):
//   Wp[n,k] = fp16(gamma[k] W[n,k]),  c1[n] = sum_k Wp[n,k] (fp32),  c0[n] = sum_k beta[k] W[n,k] + bias[n]
// gamma / beta NULL = identity LayerNorm (layer 0 consumes the already normalised embeddings)
__global__ void pack_defer_kernel(const float *__restrict__ W, const float *__restrict__ bias, const float *__restrict__ gamma,
                                  const float *__restrict__ beta, int N, int K, __half *__restrict__ Wp, float *__restrict__ c1,
                                  float *__restrict__ c0) {
    const int n = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (n >= N) return;
    float s1 = 0.f, s0 = 0.f;
    for (int k = lane; k < K; k += 32) {
        const float w = W[static_cast<int64_t>(n) * K + k];
        const __half h = __float2half_rn(gamma ? gamma[k] * w : w);
        Wp[static_cast<int64_t>(n) * K + k] = h;
        s1 += __half2float(h);
        s0 = fmaf(beta ? beta[k] : 0.f, w, s0);
    }
    s1 = warp_sum(s1);
    s0 = warp_sum(s0);
    if (lane == 0) {
        c1[n] = s1;
        c0[n] = s0 + bias[n];
    }
}

// ------------------------------------------------------------------------------------------------
// elementwise / normalisation kernels (one warp per row, float4 lanes; H % 128 == 0, H <= 1024)
// ------------------------------------------------------------------------------------------------
constexpr int LN_MAXV = 8;

__device__ __forceinline__ void ln_row(float4 (&x)[LN_MAXV], int nv, int H, const float *__restrict__ w,
                                       const float *__restrict__ b, float eps, int lane, float *out_full,
                                       __half *out_half) {
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < LN_MAXV; ++i)
        if (i < nv) s += (x[i].x + x[i].y) + (x[i].z + x[i].w);
    const float mean = warp_sum(s) / static_cast<float>(H);
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < LN_MAXV; ++i)
        if (i < nv) {
            const float a = x[i].x - mean, c = x[i].y - mean, d = x[i].z - mean, e = x[i].w - mean;
            q += (a * a + c * c) + (d * d + e * e);
        }
    const float var = warp_sum(q) / static_cast<float>(H);
    const float rstd = 1.f / sqrtf(var + eps);
#pragma unroll
    for (int i = 0; i < LN_MAXV; ++i)
        if (i < nv) {
            const int col = (lane + 32 * i) * 4;
            const float4 w4 = __ldg(reinterpret_cast<const float4 *>(w + col));
            const float4 b4 = __ldg(reinterpret_cast<const float4 *>(b + col));
            float4 o;
            o.x = (x[i].x - mean) * rstd * w4.x + b4.x;
            o.y = (x[i].y - mean) * rstd * w4.y + b4.y;
            o.z = (x[i].z - mean) * rstd * w4.z + b4.z;
            o.w = (x[i].w - mean) * rstd * w4.w + b4.w;
            if (out_full) *reinterpret_cast<float4 *>(out_full + col) = o;
            if (out_half) {
                __half2 h0 = __floats2half2_rn(o.x, o.y), h1 = __floats2half2_rn(o.z, o.w);
                uint2 pk;
                pk.x = *reinterpret_cast<uint32_t *>(&h0);
                pk.y = *reinterpret_cast<uint32_t *>(&h1);
                *reinterpret_cast<uint2 *>(out_half + col) = pk;
            }
        }
}

__global__ void layernorm_kernel(const float *__restrict__ in, const float *__restrict__ w, const float *__restrict__ b,
                                 float eps, int rows, int H, float *__restrict__ out_full, __half *__restrict__ out_half) {
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= rows) return;
    const int nv = H / 128;
    float4 x[LN_MAXV];
    const float *src = in + static_cast<int64_t>(row) * H;
#pragma unroll
    for (int i = 0; i < LN_MAXV; ++i)
        if (i < nv) x[i] = *reinterpret_cast<const float4 *>(src + (lane + 32 * i) * 4);
    ln_row(x, nv, H, w, b, eps, lane, out_full ? out_full + static_cast<int64_t>(row) * H : nullptr,
           out_half ? out_half + static_cast<int64_t>(row) * H : nullptr);
}

// modeling_bert.py:53-113 / modeling_roberta.py:146-159: (word + type) + position -> LayerNorm
__global__ void embed_ln_kernel(const int32_t *__restrict__ ids, const int32_t *__restrict__ type_ids,
                                const float *__restrict__ word, const float *__restrict__ pos,
                                const float *__restrict__ type, const float *__restrict__ w,
                                const float *__restrict__ b, float eps, int B, int S, int H, int arch, int pad_idx,
                                int vocab, int max_pos, int type_vocab, float *__restrict__ out_full,
                                __half *__restrict__ out_half) {
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= B * S) return;
    const int bq = row / S, s = row % S;
    int id = ids[row];
    id = min(max(id, 0), vocab - 1);
    int tt = type_ids ? type_ids[row] : 0;
    tt = min(max(tt, 0), type_vocab - 1);
    int p = s;
    if (arch == AC_ARCH_ROBERTA) {
        // position = cumsum(ids != pad)[s] * (id != pad) + pad_idx
        int cnt = 0;
        for (int j = lane; j <= s; j += 32) cnt += (ids[bq * S + j] != pad_idx) ? 1 : 0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
        p = (id != pad_idx) ? cnt + pad_idx : pad_idx;
    }
    p = min(p, max_pos - 1);
    const int nv = H / 128;
    float4 x[LN_MAXV];
#pragma unroll
    for (int i = 0; i < LN_MAXV; ++i)
        if (i < nv) {
            const int col = (lane + 32 * i) * 4;
            const float4 a = __ldg(reinterpret_cast<const float4 *>(word + static_cast<int64_t>(id) * H + col));
            const float4 t = __ldg(reinterpret_cast<const float4 *>(type + static_cast<int64_t>(tt) * H + col));
            const float4 q = __ldg(reinterpret_cast<const float4 *>(pos + static_cast<int64_t>(p) * H + col));
            x[i].x = (a.x + t.x) + q.x;
            x[i].y = (a.y + t.y) + q.y;
            x[i].z = (a.z + t.z) + q.z;
            x[i].w = (a.w + t.w) + q.w;
        }
    ln_row(x, nv, H, w, b, eps, lane, out_full + static_cast<int64_t>(row) * H, out_half + static_cast<int64_t>(row) * H);
}

// classifier.py:1272,1275: CLS row -> x / max(||x||_2, 1e-12)
__global__ void cls_normalize_kernel(const float *__restrict__ x, int B, int S, int H, float *__restrict__ out) {
    const int bq = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (bq >= B) return;
    const float *src = x + static_cast<int64_t>(bq) * S * H;
    float s = 0.f;
    for (int i = lane; i < H; i += 32) s = fmaf(src[i], src[i], s);
    const float nrm = fmaxf(sqrtf(warp_sum(s)), 1e-12f);
    for (int i = lane; i < H; i += 32) out[static_cast<int64_t>(bq) * H + i] = src[i] / nrm;
}

// last layer: only the CLS row of every sequence is needed downstream of attention (classifier.py:1272), so the
// output projection, both LayerNorms and the FFN of the last layer run on B rows instead of B*S
__global__ void gather_cls_kernel(const __half *__restrict__ ctx, const float *__restrict__ x, int B, int S, int H,
                                  __half *__restrict__ ctx_cls, float *__restrict__ x_cls) {
    const int bq = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (bq >= B) return;
    const int64_t src = static_cast<int64_t>(bq) * S * H, dst = static_cast<int64_t>(bq) * H;
    for (int i = lane; i < H / 8; i += 32)
        reinterpret_cast<uint4 *>(ctx_cls + dst)[i] = reinterpret_cast<const uint4 *>(ctx + src)[i];
    for (int i = lane; i < H / 4; i += 32)
        reinterpret_cast<float4 *>(x_cls + dst)[i] = reinterpret_cast<const float4 *>(x + src)[i];
}

__global__ void round_copy_kernel(const float *__restrict__ in, float *__restrict__ out, int64_t n, int do_round) {
    const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
    for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride)
        out[i] = do_round ? round_tf32(in[i]) : in[i];
}
__global__ void to_half_kernel(const float *__restrict__ in, __half *__restrict__ out, int64_t n) {
    const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
    for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride)
        out[i] = __float2half_rn(in[i]);
}

// ------------------------------------------------------------------------------------------------
// attention: one CTA (128 threads) per (sequence b, head h); S <= 128, head_dim == 64, fp16 operands.
//   scores[128x128] = Q K^T        4 x tcgen05.mma kind::f16 (M128 N128 K16), accumulator TMEM cols [0,128)
//   P = exp(scale*(s - max)) masked  thread = query row, tcgen05.ld 32x32b; P -> smem (swizzled fp16)
//   out[128x64] = P V              8 x tcgen05.mma (M128 N64 K16), accumulator TMEM cols [0,64) (scores already drained)
//   ctx[row, h*64 + :] = out / rowsum  (fp16: the A operand of the output projection)
// smem: Q tile 16 KB | K tile 16 KB (TMA, 128B swizzle), reused for P (2 slabs x 16 KB); V^T 2 slabs x 8 KB by TMA
// from the transposed buffer the QKV epilogue wrote.  48 KB + 128 TMEM columns per CTA -> 4 CTAs per SM.
// ------------------------------------------------------------------------------------------------
constexpr int ATT_THREADS = 128;
constexpr int ATT_SMEM = 48 * 1024 + 1024 /*align*/ + 64;
constexpr int ATT_TMEM_COLS = 128;

// bits lo..hi (clamped to 0..31) of a 32-key mask word: the keys of the word inside a query row's window
__device__ __forceinline__ uint32_t window_bits(int lo, int hi) {
    lo = max(lo, 0);
    hi = min(hi, 31);
    if (lo > hi) return 0u;
    const uint32_t upto = (hi == 31) ? 0xffffffffu : ((1u << (hi + 1)) - 1u);
    return upto & ~((1u << lo) - 1u);
}

// WIN (ModernBERT sliding layers, modeling_modernbert.py:262 / masking_utils.py:121-131): key k is visible to query q only
// when |q - k| <= window (inclusive).  The window is folded into each query row's key bitmask, so a row whose window holds
// no valid key ends with sum = 0 and writes zeros (never NaN / Inf).
template <bool WIN>
__global__ void __launch_bounds__(ATT_THREADS)
attention_kernel(const __grid_constant__ CUtensorMap tmap_qk, const __grid_constant__ CUtensorMap tmap_vt,
                 const int32_t *__restrict__ mask, int B, int S, int heads, int H, __half *__restrict__ ctx, int window) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t *smem = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t *sQ = smem;                    // [128 rows x 128 B]
    uint8_t *sK = smem + 16 * 1024;        // [128 rows x 128 B]
    uint8_t *sP = smem;                    // 2 slabs x [128 rows x 128 B (64 keys)]   (after QK^T retired)
    uint8_t *sVt = smem + 32 * 1024;       // 2 slabs x [64 rows (d) x 128 B (64 keys)]
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem + 48 * 1024);
    uint64_t *bar_load = bars, *bar_s = bars + 1, *bar_o = bars + 2;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 3);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int b = blockIdx.x / heads, h = blockIdx.x % heads;
    const int64_t row0 = static_cast<int64_t>(b) * S;

    if (tid == 0) {
        tma_prefetch_desc(&tmap_qk);
        tma_prefetch_desc(&tmap_vt);
        mbar_init(bar_load, 1);
        mbar_init(bar_s, 1);
        mbar_init(bar_o, 1);
        fence_mbar_init();
    }
    if (warp == 0) {
        tmem_alloc(tmem_slot, ATT_TMEM_COLS);
        tmem_relinquish();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (tid == 0) {
        mbar_arrive_expect_tx(bar_load, 48 * 1024);
        const int r = static_cast<int>(row0);
        tma_load_2d(sQ, &tmap_qk, bar_load, h * 64, r);
        tma_load_2d(sK, &tmap_qk, bar_load, H + h * 64, r);
        const int vrow = (b * heads + h) * 64;                 // rows (b, h, d) of the transposed V buffer
        tma_load_2d(sVt, &tmap_vt, bar_load, 0, vrow);
        tma_load_2d(sVt + 8 * 1024, &tmap_vt, bar_load, 64, vrow);
        // ---- S = Q K^T
        mbar_wait_guarded(bar_load, 0);
        tc_fence_after();
        constexpr uint32_t idesc_s = umma_idesc(0 /*f16*/, 128, 128);
        const uint64_t a = umma_desc_sw128(smem_u32(sQ));
        const uint64_t bdesc = umma_desc_sw128(smem_u32(sK));
#pragma unroll
        for (int k = 0; k < 4; ++k) umma_f16(tmem_base, a + 2 * k, bdesc + 2 * k, idesc_s, k != 0);
        tc_commit(bar_s);
    }
    __syncwarp();
    mbar_wait_guarded(bar_s, 0);
    tc_fence_after();

    // ---- softmax: thread = query row (TMEM lane), two passes over the 128 score columns
    const int qrow = warp * 32 + lane;
    const uint32_t t_s = tmem_base + (static_cast<uint32_t>(warp * 32) << 16);
    // key validity (key < S and not padded) as four 32-bit words held by every thread: lane l of a warp tests key
    // 32*w + l once, ballots, and the loops below only test bits
    uint32_t kmask[4];
#pragma unroll
    for (int w4 = 0; w4 < 4; ++w4) {
        const int key = 32 * w4 + lane;
        const bool ok = (key < S) && (!mask || mask[row0 + key] != 0);
        kmask[w4] = __ballot_sync(0xffffffffu, ok);
    }
    if (WIN) {
#pragma unroll
        for (int w4 = 0; w4 < 4; ++w4) kmask[w4] &= window_bits(qrow - window - 32 * w4, qrow + window - 32 * w4);
    }
    const float scale_log2 = rsqrtf(64.f) * 1.44269504088896340736f;
    float mx = -CUDART_INF_F;
#pragma unroll 1
    for (int c = 0; c < 128; c += 32) {
        uint32_t r[32];
        tmem_ld_32x32(t_s + c, r);
        tmem_ld_wait();
        const uint32_t km = c == 0 ? kmask[0] : c == 32 ? kmask[1] : c == 64 ? kmask[2] : kmask[3];
#pragma unroll
        for (int j = 0; j < 32; ++j)
            if ((km >> j) & 1u) mx = fmaxf(mx, __uint_as_float(r[j]));
    }
    float sum = 0.f;
    const uint32_t sp_base = smem_u32(sP);
#pragma unroll 1
    for (int c = 0; c < 128; c += 32) {
        uint32_t r[32];
        tmem_ld_32x32(t_s + c, r);
        tmem_ld_wait();
        uint32_t pk[16];
        const uint32_t km = c == 0 ? kmask[0] : c == 32 ? kmask[1] : c == 64 ? kmask[2] : kmask[3];
        const float mxs = mx * scale_log2;
#pragma unroll
        for (int j = 0; j < 32; j += 2) {
            const float e0 = ((km >> j) & 1u) ? ex2_approx(fmaf(__uint_as_float(r[j]), scale_log2, -mxs)) : 0.f;
            const float e1 = ((km >> (j + 1)) & 1u) ? ex2_approx(fmaf(__uint_as_float(r[j + 1]), scale_log2, -mxs)) : 0.f;
            sum += e0 + e1;
            __half2 hh = __floats2half2_rn(e0, e1);
            pk[j >> 1] = *reinterpret_cast<uint32_t *>(&hh);
        }
        // slab (c / 64), row qrow: 4 x 16-byte chunks (8 keys each) starting at chunk (c % 64) / 8
        const uint32_t prow = sp_base + (c >> 6) * 16384 + (qrow >> 3) * 1024 + (qrow & 7) * 128;
        const int ch0 = (c & 63) >> 3;
#pragma unroll
        for (int ch = 0; ch < 4; ++ch) {
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(prow + (((ch0 + ch) ^ (qrow & 7)) << 4)),
                         "r"(pk[4 * ch]), "r"(pk[4 * ch + 1]), "r"(pk[4 * ch + 2]), "r"(pk[4 * ch + 3])
                         : "memory");
        }
    }
    // generic-proxy smem writes (P) -> visible to the tensor-core (async) proxy; all threads are done reading S
    fence_proxy_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();

    // ---- O = P V   (accumulates into TMEM columns [0,64): the score tile is dead)
    if (tid == 0) {
        constexpr uint32_t idesc_o = umma_idesc(0 /*f16*/, 128, 64);
#pragma unroll
        for (int slab = 0; slab < 2; ++slab) {
            const uint64_t a = umma_desc_sw128(smem_u32(sP + slab * 16384));
            const uint64_t bdesc = umma_desc_sw128(smem_u32(sVt + slab * 8192));
#pragma unroll
            for (int k = 0; k < 4; ++k) umma_f16(tmem_base, a + 2 * k, bdesc + 2 * k, idesc_o, (slab | k) != 0);
        }
        tc_commit(bar_o);
    }
    __syncwarp();
    mbar_wait_guarded(bar_o, 0);
    tc_fence_after();

    const float inv = (sum > 0.f) ? 1.f / sum : 0.f;
#pragma unroll 1
    for (int c = 0; c < 64; c += 32) {
        uint32_t r[32];
        tmem_ld_32x32(t_s + c, r);
        tmem_ld_wait();
        if (qrow < S) {
            __half *dst = ctx + (row0 + qrow) * H + h * 64 + c;
#pragma unroll
            for (int j = 0; j < 32; j += 8) {
                __half2 h0 = __floats2half2_rn(__uint_as_float(r[j]) * inv, __uint_as_float(r[j + 1]) * inv);
                __half2 h1 = __floats2half2_rn(__uint_as_float(r[j + 2]) * inv, __uint_as_float(r[j + 3]) * inv);
                __half2 h2 = __floats2half2_rn(__uint_as_float(r[j + 4]) * inv, __uint_as_float(r[j + 5]) * inv);
                __half2 h3 = __floats2half2_rn(__uint_as_float(r[j + 6]) * inv, __uint_as_float(r[j + 7]) * inv);
                uint4 pk;
                pk.x = *reinterpret_cast<uint32_t *>(&h0); pk.y = *reinterpret_cast<uint32_t *>(&h1);
                pk.z = *reinterpret_cast<uint32_t *>(&h2); pk.w = *reinterpret_cast<uint32_t *>(&h3);
                *reinterpret_cast<uint4 *>(dst + j) = pk;
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
        tc_fence_after();
        tmem_dealloc(tmem_base, ATT_TMEM_COLS);
    }
}

// ------------------------------------------------------------------------------------------------
// attention for 128 < S <= 512: one CTA per (sequence, head, 128-query block), key blocks of 128 streamed twice.
//   pass A  row max over all key blocks        (QK^T only)
//   pass B  P = exp(scale*(s - max)) per block, O += P V_block accumulated in TMEM, row sums in registers
// Using the final max in pass B means the TMEM accumulator never has to be rescaled; the price is computing QK^T
// twice (QK^T is half of the attention flops, attention is ~3 % of the encoder).  Serial per block (TMA -> MMA ->
// softmax -> MMA); the S <= 128 kernel above is the tuned path of the benchmark configurations.
// ------------------------------------------------------------------------------------------------
constexpr int ATTL_SMEM = 80 * 1024 + 1024 + 64;
constexpr int ATTL_TMEM_COLS = 256;

// WIN: the same per-row key window as attention_kernel; key blocks that lie entirely outside the window of every query of
// this 128-query block are skipped (never loaded, never multiplied).
template <bool WIN>
__global__ void __launch_bounds__(ATT_THREADS)
attention_long_kernel(const __grid_constant__ CUtensorMap tmap_qk, const __grid_constant__ CUtensorMap tmap_vt,
                      const int32_t *__restrict__ mask, int B, int S, int heads, int H, __half *__restrict__ ctx, int window) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t *smem = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t *sQ = smem;                    // [128 x 128 B]
    uint8_t *sK = smem + 16 * 1024;        // [128 x 128 B] current key block
    uint8_t *sVt = smem + 32 * 1024;       // 2 slabs x [64 (d) x 128 B (64 keys)]
    uint8_t *sP = smem + 48 * 1024;        // 2 slabs x [128 x 128 B (64 keys)]
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem + 80 * 1024);
    uint64_t *bar_load = bars, *bar_s = bars + 1, *bar_o = bars + 2;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 3);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int b = blockIdx.x / heads, h = blockIdx.x % heads;
    const int qb = blockIdx.y;                                   // query block
    const int nkb = (S + 127) / 128;
    const int64_t row0 = static_cast<int64_t>(b) * S;
    const int vrow = (b * heads + h) * 64;
    // key blocks [jlo, jend) can hold a visible key of this query block
    const int jlo = WIN ? max(qb * 128 - window, 0) / 128 : 0;
    const int jend = WIN ? min((min(qb * 128 + 127, S - 1) + window) / 128 + 1, nkb) : nkb;

    if (tid == 0) {
        tma_prefetch_desc(&tmap_qk);
        tma_prefetch_desc(&tmap_vt);
        mbar_init(bar_load, 1);
        mbar_init(bar_s, 1);
        mbar_init(bar_o, 1);
        fence_mbar_init();
    }
    if (warp == 0) {
        tmem_alloc(tmem_slot, ATTL_TMEM_COLS);
        tmem_relinquish();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const uint32_t t_s = tmem_base + (static_cast<uint32_t>(warp * 32) << 16);
    const int qrow = warp * 32 + lane;                            // row inside the query block
    const int qglob = qb * 128 + qrow;                            // position inside the sequence
    const float scale_log2 = rsqrtf(64.f) * 1.44269504088896340736f;
    constexpr uint32_t idesc_s = umma_idesc(0, 128, 128);
    constexpr uint32_t idesc_o = umma_idesc(0, 128, 64);

    uint32_t ph_load = 0, ph_s = 0, ph_o = 0;
    float mx = -CUDART_INF_F, sum = 0.f;

    for (int pass = 0; pass < 2; ++pass) {
        for (int j = jlo; j < jend; ++j) {
            const int key0 = j * 128;
            if (tid == 0) {
                const bool first = (pass == 0 && j == jlo);
                const uint32_t bytes = (first ? 16 * 1024 : 0) + 16 * 1024 + (pass == 1 ? 16 * 1024 : 0);
                mbar_arrive_expect_tx(bar_load, bytes);
                if (first) tma_load_2d(sQ, &tmap_qk, bar_load, h * 64, static_cast<int>(row0) + qb * 128);
                tma_load_2d(sK, &tmap_qk, bar_load, H + h * 64, static_cast<int>(row0) + key0);
                if (pass == 1) {
                    tma_load_2d(sVt, &tmap_vt, bar_load, key0, vrow);
                    tma_load_2d(sVt + 8 * 1024, &tmap_vt, bar_load, key0 + 64, vrow);
                }
                mbar_wait_guarded(bar_load, ph_load);
                tc_fence_after();
                const uint64_t a = umma_desc_sw128(smem_u32(sQ));
                const uint64_t bd = umma_desc_sw128(smem_u32(sK));
#pragma unroll
                for (int k = 0; k < 4; ++k) umma_f16(tmem_base, a + 2 * k, bd + 2 * k, idesc_s, k != 0);
                tc_commit(bar_s);
            }
            ph_load ^= 1;
            __syncwarp();
            mbar_wait_guarded(bar_s, ph_s);
            ph_s ^= 1;
            tc_fence_after();

            // key validity bits of this block
            uint32_t kmask[4];
#pragma unroll
            for (int w4 = 0; w4 < 4; ++w4) {
                const int key = key0 + 32 * w4 + lane;
                const bool ok = (key < S) && (!mask || mask[row0 + key] != 0);
                kmask[w4] = __ballot_sync(0xffffffffu, ok);
            }
            if (WIN) {
#pragma unroll
                for (int w4 = 0; w4 < 4; ++w4) {
                    const int k0 = key0 + 32 * w4;
                    kmask[w4] &= window_bits(qglob - window - k0, qglob + window - k0);
                }
            }
            if (pass == 0) {
#pragma unroll
                for (int ci = 0; ci < 4; ++ci) {
                    uint32_t r[32];
                    tmem_ld_32x32(t_s + 32 * ci, r);
                    tmem_ld_wait();
                    const uint32_t km = kmask[ci];
#pragma unroll
                    for (int jj = 0; jj < 32; ++jj)
                        if ((km >> jj) & 1u) mx = fmaxf(mx, __uint_as_float(r[jj]));
                }
                tc_fence_before();
                __syncthreads();                                  // S columns and sK may be overwritten now
                tc_fence_after();
            } else {
                const uint32_t sp_base = smem_u32(sP);
                const float mxs = mx * scale_log2;
#pragma unroll
                for (int ci = 0; ci < 4; ++ci) {
                    const int c = 32 * ci;
                    uint32_t r[32];
                    tmem_ld_32x32(t_s + c, r);
                    tmem_ld_wait();
                    const uint32_t km = kmask[ci];
                    uint32_t pk[16];
#pragma unroll
                    for (int jj = 0; jj < 32; jj += 2) {
                        const float e0 = ((km >> jj) & 1u) ? ex2_approx(fmaf(__uint_as_float(r[jj]), scale_log2, -mxs)) : 0.f;
                        const float e1 = ((km >> (jj + 1)) & 1u) ? ex2_approx(fmaf(__uint_as_float(r[jj + 1]), scale_log2, -mxs)) : 0.f;
                        sum += e0 + e1;
                        __half2 hh = __floats2half2_rn(e0, e1);
                        pk[jj >> 1] = *reinterpret_cast<uint32_t *>(&hh);
                    }
                    const uint32_t prow = sp_base + (c >> 6) * 16384 + (qrow >> 3) * 1024 + (qrow & 7) * 128;
                    const int ch0 = (c & 63) >> 3;
#pragma unroll
                    for (int ch = 0; ch < 4; ++ch) {
                        asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(prow + (((ch0 + ch) ^ (qrow & 7)) << 4)),
                                     "r"(pk[4 * ch]), "r"(pk[4 * ch + 1]), "r"(pk[4 * ch + 2]), "r"(pk[4 * ch + 3])
                                     : "memory");
                    }
                }
                fence_proxy_async_smem();
                tc_fence_before();
                __syncthreads();
                tc_fence_after();
                if (tid == 0) {
#pragma unroll
                    for (int slab = 0; slab < 2; ++slab) {
                        const uint64_t a = umma_desc_sw128(smem_u32(sP + slab * 16384));
                        const uint64_t bd = umma_desc_sw128(smem_u32(sVt + slab * 8192));
#pragma unroll
                        for (int k = 0; k < 4; ++k)
                            umma_f16(tmem_base + 128, a + 2 * k, bd + 2 * k, idesc_o, ((WIN ? j - jlo : j) | slab | k) != 0);
                    }
                    tc_commit(bar_o);
                }
                __syncwarp();
                mbar_wait_guarded(bar_o, ph_o);                   // sK / sVt / sP / S columns are free again
                ph_o ^= 1;
                tc_fence_after();
            }
        }
    }

    const float inv = (sum > 0.f) ? 1.f / sum : 0.f;
#pragma unroll 1
    for (int c = 0; c < 64; c += 32) {
        uint32_t r[32];
        tmem_ld_32x32(t_s + 128 + c, r);
        tmem_ld_wait();
        if (qglob < S) {
            __half *dst = ctx + (row0 + qglob) * H + h * 64 + c;
#pragma unroll
            for (int jj = 0; jj < 32; jj += 8) {
                __half2 h0 = __floats2half2_rn(__uint_as_float(r[jj]) * inv, __uint_as_float(r[jj + 1]) * inv);
                __half2 h1 = __floats2half2_rn(__uint_as_float(r[jj + 2]) * inv, __uint_as_float(r[jj + 3]) * inv);
                __half2 h2 = __floats2half2_rn(__uint_as_float(r[jj + 4]) * inv, __uint_as_float(r[jj + 5]) * inv);
                __half2 h3 = __floats2half2_rn(__uint_as_float(r[jj + 6]) * inv, __uint_as_float(r[jj + 7]) * inv);
                uint4 pk;
                pk.x = *reinterpret_cast<uint32_t *>(&h0); pk.y = *reinterpret_cast<uint32_t *>(&h1);
                pk.z = *reinterpret_cast<uint32_t *>(&h2); pk.w = *reinterpret_cast<uint32_t *>(&h3);
                *reinterpret_cast<uint4 *>(dst + jj) = pk;
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
        tc_fence_after();
        tmem_dealloc(tmem_base, ATTL_TMEM_COLS);
    }
}

// last layer, deferred flow: CLS rows of the attention context and of LN_pending(y) (two-pass statistics from the fp32 sums)
__global__ void gather_cls_ln_kernel(const __half *__restrict__ ctx, const float *__restrict__ y, int B, int S, int H,
                                     const float *__restrict__ g, const float *__restrict__ b, float eps,
                                     __half *__restrict__ ctx_cls, float *__restrict__ x_cls) {
    const int bq = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (bq >= B) return;
    const int64_t src = static_cast<int64_t>(bq) * S * H, dst = static_cast<int64_t>(bq) * H;
    for (int i = lane; i < H / 8; i += 32)
        reinterpret_cast<uint4 *>(ctx_cls + dst)[i] = reinterpret_cast<const uint4 *>(ctx + src)[i];
    const int nv = H / 128;
    float4 x[LN_MAXV];
#pragma unroll
    for (int i = 0; i < LN_MAXV; ++i)
        if (i < nv) x[i] = *reinterpret_cast<const float4 *>(y + src + (lane + 32 * i) * 4);
    ln_row(x, nv, H, g, b, eps, lane, x_cls + dst, nullptr);
}

// ================================================================================================
// ModernBERT (HF modeling_modernbert.py): pre-LN blocks, RoPE attention with per-layer windows, GeGLU FFN
// ================================================================================================

// modeling_modernbert.py:52-71: LayerNorm(tok_embeddings[ids]); no position or token-type rows
__global__ void embed_norm_kernel(const int32_t *__restrict__ ids, const float *__restrict__ tok, const float *__restrict__ w,
                                  const float *__restrict__ b, float eps, int rows, int H, int vocab, float *__restrict__ out_full,
                                  __half *__restrict__ out_half) {
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= rows) return;
    const int id = min(max(ids[row], 0), vocab - 1);
    const int nv = H / 128;
    float4 x[LN_MAXV];
#pragma unroll
    for (int i = 0; i < LN_MAXV; ++i)
        if (i < nv) x[i] = __ldg(reinterpret_cast<const float4 *>(tok + static_cast<int64_t>(id) * H + (lane + 32 * i) * 4));
    ln_row(x, nv, H, w, b, eps, lane, out_full + static_cast<int64_t>(row) * H, out_half + static_cast<int64_t>(row) * H);
}

// 32 fp32 values of one accumulator row -> fp16 Y[row_base + lane, col0 .. col0 + 32) through the warp's staging tile
// (the store pattern of EpiLinear's fp16 path: 8 rows x 4 x 16 B per pass)
__device__ __forceinline__ void store_row32_half(const float (&y)[32], uint8_t *stage, int lane, int row_base, int col0, int M,
                                                 int N, int ldy, __half *Y) {
    uint4 *srow = reinterpret_cast<uint4 *>(stage + lane * GEMM_EPI_STAGE_ROW_BYTES);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        uint4 pk;
        __half2 h0 = __floats2half2_rn(y[8 * j], y[8 * j + 1]), h1 = __floats2half2_rn(y[8 * j + 2], y[8 * j + 3]);
        __half2 h2 = __floats2half2_rn(y[8 * j + 4], y[8 * j + 5]), h3 = __floats2half2_rn(y[8 * j + 6], y[8 * j + 7]);
        pk.x = *reinterpret_cast<uint32_t *>(&h0); pk.y = *reinterpret_cast<uint32_t *>(&h1);
        pk.z = *reinterpret_cast<uint32_t *>(&h2); pk.w = *reinterpret_cast<uint32_t *>(&h3);
        srow[j] = pk;
    }
    __syncwarp();
    const int r8 = lane >> 2, c = lane & 3;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int rr = r8 + 8 * i;
        const int grow = row_base + rr;
        const int col = col0 + 8 * c;
        if (grow < M && col + 8 <= N) {
            const uint4 pk = *reinterpret_cast<const uint4 *>(stage + rr * GEMM_EPI_STAGE_ROW_BYTES + 16 * c);
            *reinterpret_cast<uint4 *>(Y + static_cast<int64_t>(grow) * ldy + col) = pk;
        }
    }
    __syncwarp();
}

// fused Wqkv epilogue (modeling_modernbert.py:285-296): acc + bias, RoPE on the q and k thirds in fp32 before the fp16
// rounding, V third written transposed as EpiLinear's VT path does.  One epilogue warp drains 128 columns (two whole heads)
// in 32-column chunks, so the thread holding head columns d = 0..31 of its row receives d = 32..63 in the next chunk: the
// first half waits in registers, the second chunk rotates both (rotate_half pairs d with d + 32) and stores 64 columns.
//   q'[d]      = q[d] cos - q[d + 32] sin        q'[d + 32] = q[d + 32] cos + q[d] sin       (cos, sin of angle pos * f_d)
// cs: [512 positions][32] (cos, sin) for this layer's theta, position = row % S (position_ids = arange(S)).
struct EpiQKVRope {
    const float *__restrict__ bias;       // [3H]
    __half *qk;                           // [M, 2H] rotated q | k
    __half *vT;                           // [(b, feature), S_pad] V^T
    const float2 *__restrict__ cs;        // [512, 32]
    int M, H, S, S_pad;

    static constexpr int kUnrollChunks = 4;
    static constexpr int kPrefetchDist = 1;
    struct State {
        float lo[32];                     // head columns 0..31 (acc + bias) of the chunk drained before
    };
    __device__ __forceinline__ void begin_cta(State &, int, int) const {}
    __device__ __forceinline__ void end_cta(State &, int, int) const {}
    __device__ __forceinline__ void prefetch(State &, const GemmTileInfo &, int, int, int, int) const {}

    __device__ __forceinline__ void tile(State &st, const GemmTileInfo &ti, int row, int col0, const float (&v)[32],
                                         uint8_t *stage, int lane, int, uint32_t) const {
        const int row_base = ti.m0 + ((threadIdx.x >> 5) & 3) * 32;
        if (row_base >= M || col0 >= 3 * H) return;                        // warp-uniform
        if (col0 >= 2 * H) {
            if (row < M) {
                const int b = row / S, key = row - b * S;
                __half *dst = vT + (static_cast<int64_t>(b) * H + (col0 - 2 * H)) * S_pad + key;
#pragma unroll
                for (int j = 0; j < 32; j += 4) {
                    const float4 b4 = __ldg(reinterpret_cast<const float4 *>(bias + col0 + j));
                    dst[static_cast<int64_t>(j) * S_pad] = __float2half_rn(v[j] + b4.x);
                    dst[static_cast<int64_t>(j + 1) * S_pad] = __float2half_rn(v[j + 1] + b4.y);
                    dst[static_cast<int64_t>(j + 2) * S_pad] = __float2half_rn(v[j + 2] + b4.z);
                    dst[static_cast<int64_t>(j + 3) * S_pad] = __float2half_rn(v[j + 3] + b4.w);
                }
            }
            return;
        }
        if ((col0 & 32) == 0) {                                              // head columns 0..31: keep for the next chunk
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
                const float4 b4 = __ldg(reinterpret_cast<const float4 *>(bias + col0 + j));
                st.lo[j] = v[j] + b4.x; st.lo[j + 1] = v[j + 1] + b4.y;
                st.lo[j + 2] = v[j + 2] + b4.z; st.lo[j + 3] = v[j + 3] + b4.w;
            }
            return;
        }
        const int pos = (row < M) ? row % S : 0;
        const float4 *cs4 = reinterpret_cast<const float4 *>(cs + pos * 32);   // (cos, sin) of d, d + 1
        // both halves in one pass: the rotated first half overwrites st.lo, the second half goes to hi (peak 64 live values)
        float hi[32];
#pragma unroll
        for (int j = 0; j < 32; j += 2) {
            const float4 t = __ldg(cs4 + (j >> 1));
            const float2 b2 = __ldg(reinterpret_cast<const float2 *>(bias + col0 + j));
            const float h0 = v[j] + b2.x, h1 = v[j + 1] + b2.y;
            const float l0 = st.lo[j], l1 = st.lo[j + 1];
            st.lo[j] = fmaf(l0, t.x, -h0 * t.y);
            st.lo[j + 1] = fmaf(l1, t.z, -h1 * t.w);
            hi[j] = fmaf(h0, t.x, l0 * t.y);
            hi[j + 1] = fmaf(h1, t.z, l1 * t.w);
        }
        store_row32_half(st.lo, stage, lane, row_base, col0 - 32, M, 2 * H, 2 * H, qk);
        store_row32_half(hi, stage, lane, row_base, col0, M, 2 * H, 2 * H, qk);
    }
};

// GeGLU FFN1 epilogue (modeling_modernbert.py:88-91): Wi is packed at create time so that accumulator chunk q (32 columns)
// holds input columns 16q .. 16q+15 followed by the matching gate columns I + 16q ..; the thread of a row writes
// gelu_erf(input + b) * (gate + b') as 16 fp16 values (one 32-byte sector) at output columns 16q .. 16q+15 of Y[M, I].
// Chunks at or past N = 2I are skipped (the last 256-column tile of ModernBERT-large's 2I = 5248 is half empty).
struct EpiGeGLU {
    const float *__restrict__ bias;       // [2I] in packed order
    __half *Y;                            // [M, I]
    int M, N, I;

    static constexpr int kUnrollChunks = 4;
    static constexpr int kPrefetchDist = 1;
    struct State {};
    __device__ __forceinline__ void begin_cta(State &, int, int) const {}
    __device__ __forceinline__ void end_cta(State &, int, int) const {}
    __device__ __forceinline__ void prefetch(State &, const GemmTileInfo &, int, int, int, int) const {}

    __device__ __forceinline__ void tile(State &, const GemmTileInfo &, int row, int col0, const float (&v)[32], uint8_t *,
                                         int, int, uint32_t) const {
        if (row >= M || col0 >= N) return;
        uint32_t pk[8];
#pragma unroll
        for (int j = 0; j < 16; j += 4) {
            const float4 ba = __ldg(reinterpret_cast<const float4 *>(bias + col0 + j));
            const float4 bg = __ldg(reinterpret_cast<const float4 *>(bias + col0 + 16 + j));
            const __half2 h0 = __floats2half2_rn(gelu_erf(v[j] + ba.x) * (v[16 + j] + bg.x),
                                                 gelu_erf(v[j + 1] + ba.y) * (v[17 + j] + bg.y));
            const __half2 h1 = __floats2half2_rn(gelu_erf(v[j + 2] + ba.z) * (v[18 + j] + bg.z),
                                                 gelu_erf(v[j + 3] + ba.w) * (v[19 + j] + bg.w));
            pk[j >> 1] = *reinterpret_cast<const uint32_t *>(&h0);
            pk[(j >> 1) + 1] = *reinterpret_cast<const uint32_t *>(&h1);
        }
        uint4 *dst = reinterpret_cast<uint4 *>(Y + static_cast<int64_t>(row) * I + (col0 >> 1));
        dst[0] = make_uint4(pk[0], pk[1], pk[2], pk[3]);
        dst[1] = make_uint4(pk[4], pk[5], pk[6], pk[7]);
    }
};

// Wi [2I, H] (fp32, HF rows: input 0..I-1, gate I..2I-1) -> fp16 rows in the chunk order EpiGeGLU reads, bias likewise
// (NULL bias = zeros).  Packed row p = 32 q + j: input row 16 q + j (j < 16) or gate row I + 16 q + j - 16.
__global__ void pack_geglu_kernel(const float *__restrict__ W, const float *__restrict__ bias, int I, int K, __half *__restrict__ Wp,
                                  float *__restrict__ bp) {
    const int p = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (p >= 2 * I) return;
    const int q = p >> 5, j = p & 31;
    const int src = (j < 16) ? 16 * q + j : I + 16 * q + (j - 16);
    for (int k = lane; k < K; k += 32)
        Wp[static_cast<int64_t>(p) * K + k] = __float2half_rn(W[static_cast<int64_t>(src) * K + k]);
    if (lane == 0) bp[p] = bias ? bias[src] : 0.f;
}

}  // namespace ac

// ================================================================================================
// encoder handle
// ================================================================================================
using namespace ac;

struct ac_encoder {
    ac_encoder_config cfg;
    // packed weights (device): fp16 GEMM operands, fp32 everything else
    float *word = nullptr, *pos = nullptr, *type = nullptr, *emb_ln_w = nullptr, *emb_ln_b = nullptr;
    // QKV / FFN1 consume un-normalised residual sums: their weights are packed as fp16(gamma * W) with the rank-1 correction
    // vectors c1 (row sums of the packed weight) and c0 (W beta + bias), see pack_defer_kernel
    std::vector<__half *> wqkv_d, wo, w1_d, w2;
    std::vector<float *> c1qkv, c0qkv, c1f, c0f, bo, ln1w, ln1b, b2, ln2w, ln2b;
    __half *w1_last = nullptr;            // plain fp16 FFN1 weight of the last layer (CLS-only tail runs on materialised LayerNorm rows)
    float *b1_last = nullptr;
    // activations: fp32 residual sums x (+ tmp for a materialised final LayerNorm); fp16 GEMM operands xh, qk, vT, ctx, ffn
    float *x = nullptr, *tmp = nullptr;
    __half *xh = nullptr, *qk = nullptr, *vT = nullptr, *ctx = nullptr, *ffn = nullptr;
    size_t T = 0;           // token capacity (multiple of 128)
    size_t vt_elems = 0;
    // compact CLS-row buffers of the last layer (Bc rows)
    size_t Bc = 0;
    float *x_cls = nullptr, *tmp_cls = nullptr;
    __half *xh_cls = nullptr, *ctx_cls = nullptr, *ffn_cls = nullptr;
    CUtensorMap m_xh_cls, m_ctx_cls, m_ffn_cls;
    // cached TMA descriptors: A operands (128-row boxes) and weights (128-row boxes = the B half one CTA of a pair stages)
    CUtensorMap m_xh, m_ctx, m_ffn, m_qk_att, m_vt_att;
    int vt_B = -1, vt_S = -1;
    std::vector<CUtensorMap> p_wqkv_d, p_wo, p_w1_d, p_w2;
    CUtensorMap p_w1_last;
    // row statistics (ping-pong) and the per-128-column partials the residual epilogues write
    float2 *stats_a = nullptr, *stats_b = nullptr, *stats_id = nullptr, *parts = nullptr;
    float *ones = nullptr, *zeros = nullptr;
    std::vector<void *> allocs;
    int last_B = 0, last_S = 0;
    bool last_cls_only = false;
    const float *last_hidden = nullptr;   // where the previous full forward left the last hidden state
    // ModernBERT (AC_ARCH_MODERNBERT): word = tok_embeddings, emb_ln_* = embeddings.norm; per layer wqkv_d = plain fp16 Wqkv,
    // wo / bo = attn.Wo, w1_d = Wi packed for EpiGeGLU, w2 / b2 = mlp.Wo (their tensor maps as above), and:
    std::vector<float *> bqkv, bi, attn_nw, attn_nb, mlp_nw, mlp_nb;   // biases (zeros when absent), LayerNorms (attn_* unused in layer 0)
    std::vector<float2 *> rope;           // per layer [512, 32] (cos, sin) of its theta
    std::vector<int> window;              // per layer key window, 0 = global
    float *final_nw = nullptr, *final_nb = nullptr;
};

static int launch_cls_normalize(const float *x, int B, int S, int H, float *out, cudaStream_t s) {
    const int wpb = 8;
    cls_normalize_kernel<<<(B + wpb - 1) / wpb, wpb * 32, 0, s>>>(x, B, S, H, out);
    AC_LAUNCH_CHECK();
    return AC_OK;
}

// softmax(Q K^T / 8 + mask) V into ctx [B*S, H]: tqk is the 128-row-box map of qk [rows, 2H], tvt the 64 x 64-box map of
// vT [(b, h, d), S_pad].  The one dispatch of the encoder and of ac_attention (S <= 128 / long kernel, window or global).
static int launch_attention(const CUtensorMap &tqk, const CUtensorMap &tvt, const int32_t *mask, int B, int S, int heads,
                            __half *ctx, cudaStream_t s, int window = 0) {
    const int H = heads * 64;
    // per-device: the attribute is a property of the (function, device) pair
    static bool att_attr[64] = {};
    int dev = 0;
    AC_CUDA(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 64 || !att_attr[dev]) {
        AC_CUDA(cudaFuncSetAttribute(attention_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, ATT_SMEM));
        AC_CUDA(cudaFuncSetAttribute(attention_long_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, ATTL_SMEM));
        AC_CUDA(cudaFuncSetAttribute(attention_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, ATT_SMEM));
        AC_CUDA(cudaFuncSetAttribute(attention_long_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, ATTL_SMEM));
        if (dev >= 0 && dev < 64) att_attr[dev] = true;
    }
    // algorithmic flops of softmax(QK^T)V at the true sequence length (the 128-wide tile does more)
    // a window that covers the whole sequence is global attention
    const bool win = window > 0 && window < S - 1;
    const int slot = prof_begin(PROF_ATTENTION, 4.0 * B * heads * static_cast<double>(S) * S * 64, 0.0, s);
    const dim3 grid_long(B * heads, (S + 127) / 128);
    if (S <= 128 && win)
        attention_kernel<true><<<B * heads, ATT_THREADS, ATT_SMEM, s>>>(tqk, tvt, mask, B, S, heads, H, ctx, window);
    else if (S <= 128)
        attention_kernel<false><<<B * heads, ATT_THREADS, ATT_SMEM, s>>>(tqk, tvt, mask, B, S, heads, H, ctx, 0);
    else if (win)
        attention_long_kernel<true><<<grid_long, ATT_THREADS, ATTL_SMEM, s>>>(tqk, tvt, mask, B, S, heads, H, ctx, window);
    else
        attention_long_kernel<false><<<grid_long, ATT_THREADS, ATTL_SMEM, s>>>(tqk, tvt, mask, B, S, heads, H, ctx, 0);
    prof_end(slot, s);
    AC_LAUNCH_CHECK();
    return AC_OK;
}

template <class T>
static int dev_alloc(ac_encoder *e, T **p, size_t elems) {
    void *q = nullptr;
    AC_CUDA(cudaMalloc(&q, elems * sizeof(T)));
    e->allocs.push_back(q);
    *p = static_cast<T *>(q);
    return AC_OK;
}

static int pack_f32(ac_encoder *e, float **dst, const float *src, size_t n) {
    int rc = dev_alloc(e, dst, n);
    if (rc) return rc;
    round_copy_kernel<<<256, 256>>>(src, *dst, static_cast<int64_t>(n), 0);
    AC_LAUNCH_CHECK();
    return AC_OK;
}
static int pack_f16(ac_encoder *e, __half **dst, const float *src, size_t n) {
    int rc = dev_alloc(e, dst, n);
    if (rc) return rc;
    to_half_kernel<<<256, 256>>>(src, *dst, static_cast<int64_t>(n));
    AC_LAUNCH_CHECK();
    return AC_OK;
}

extern "C" int ac_encoder_destroy(ac_encoder *enc) {
    if (!enc) return AC_OK;
    for (void *p : enc->allocs) cudaFree(p);
    delete enc;
    return AC_OK;
}

// activation workspace, row statistics and the A-operand tensor maps of an encoder sized by e->cfg (both architectures)
static int alloc_workspace(ac_encoder *e) {
    const int H = e->cfg.hidden, I = e->cfg.intermediate;
    const size_t T = e->T;
    int rc;
#define WS(x) do { rc = (x); if (rc) return rc; } while (0)
    WS(dev_alloc(e, &e->stats_a, T));
    WS(dev_alloc(e, &e->stats_b, T));
    WS(dev_alloc(e, &e->stats_id, T));
    WS(dev_alloc(e, &e->parts, static_cast<size_t>(H / 128) * T));
    WS(dev_alloc(e, &e->ones, H));
    WS(dev_alloc(e, &e->zeros, H));
    fill_stats_identity_kernel<<<static_cast<unsigned>((T + 255) / 256), 256>>>(e->stats_id, static_cast<int64_t>(T));
    fill_value_kernel<<<(H + 255) / 256, 256>>>(e->ones, H, 1.f);
    fill_value_kernel<<<(H + 255) / 256, 256>>>(e->zeros, H, 0.f);
    WS(check_cuda(cudaGetLastError(), "deferred-LayerNorm constants"));
    // V^T: (b, h, d) rows x S_pad keys, S_pad = roundup(S, 8) (TMA row pitch: 16 bytes).  Sized for every call forward_cls
    // accepts (B*S <= max_tokens): B*S_pad <= floor(max_tokens / S) * roundup(S, 8), largest at S = 1 (8 * max_tokens); for
    // S >= 8 it stays below 2 * max_tokens.
    e->vt_elems = 8 * static_cast<size_t>(e->cfg.max_tokens) * H;
    WS(dev_alloc(e, &e->x, T * H));
    WS(dev_alloc(e, &e->tmp, T * H));
    WS(dev_alloc(e, &e->xh, T * H));
    WS(dev_alloc(e, &e->qk, T * 2 * H));
    WS(dev_alloc(e, &e->vT, e->vt_elems));
    WS(dev_alloc(e, &e->ctx, T * H));
    WS(dev_alloc(e, &e->ffn, T * I));
    e->Bc = T < 16384 ? T : 16384;
    WS(dev_alloc(e, &e->x_cls, e->Bc * H));
    WS(dev_alloc(e, &e->tmp_cls, e->Bc * H));
    WS(dev_alloc(e, &e->xh_cls, e->Bc * H));
    WS(dev_alloc(e, &e->ctx_cls, e->Bc * H));
    WS(dev_alloc(e, &e->ffn_cls, e->Bc * I));
    WS(check_cuda(cudaMemset(e->xh_cls, 0, e->Bc * H * sizeof(__half)), "memset xh_cls"));
    WS(check_cuda(cudaMemset(e->ctx_cls, 0, e->Bc * H * sizeof(__half)), "memset ctx_cls"));
    WS(check_cuda(cudaMemset(e->ffn_cls, 0, e->Bc * I * sizeof(__half)), "memset ffn_cls"));
    WS(check_cuda(cudaMemset(e->qk, 0, T * 2 * H * sizeof(__half)), "memset qk"));
    WS(check_cuda(cudaMemset(e->vT, 0, e->vt_elems * sizeof(__half)), "memset vT"));
    WS(check_cuda(cudaMemset(e->xh, 0, T * H * sizeof(__half)), "memset xh"));
    WS(check_cuda(cudaMemset(e->ctx, 0, T * H * sizeof(__half)), "memset ctx"));
    WS(check_cuda(cudaMemset(e->ffn, 0, T * I * sizeof(__half)), "memset ffn"));
    // TMA descriptors (fp16: 64 elements = 128 bytes per box row)
    WS(make_tmap_2d(&e->m_xh, e->xh, 2, T, H, static_cast<uint64_t>(H) * 2, GEMM_BLOCK_M, 64));
    WS(make_tmap_2d(&e->m_ctx, e->ctx, 2, T, H, static_cast<uint64_t>(H) * 2, GEMM_BLOCK_M, 64));
    WS(make_tmap_2d(&e->m_ffn, e->ffn, 2, T, I, static_cast<uint64_t>(I) * 2, GEMM_BLOCK_M, 64));
    WS(make_tmap_2d(&e->m_qk_att, e->qk, 2, T, 2 * H, static_cast<uint64_t>(2 * H) * 2, 128, 64));
    WS(make_tmap_2d(&e->m_xh_cls, e->xh_cls, 2, e->Bc, H, static_cast<uint64_t>(H) * 2, GEMM_BLOCK_M, 64));
    WS(make_tmap_2d(&e->m_ctx_cls, e->ctx_cls, 2, e->Bc, H, static_cast<uint64_t>(H) * 2, GEMM_BLOCK_M, 64));
    WS(make_tmap_2d(&e->m_ffn_cls, e->ffn_cls, 2, e->Bc, I, static_cast<uint64_t>(I) * 2, GEMM_BLOCK_M, 64));
#undef WS
    return AC_OK;
}

extern "C" int ac_encoder_create(const ac_encoder_config *cfg, const ac_encoder_weights *w, ac_encoder **out) {
    AC_REQUIRE(cfg && w && out, "ac_encoder_create: null argument");
    AC_REQUIRE(cfg->precision == AC_PREC_F16, "ac_encoder_create: only AC_PREC_F16 (fp16 operands, fp32 accumulate) is implemented");
    AC_REQUIRE(cfg->hidden % 128 == 0 && cfg->hidden <= 1024, "ac_encoder_create: hidden=%d must be a multiple of 128, <= 1024", cfg->hidden);
    AC_REQUIRE(cfg->heads > 0 && cfg->hidden / cfg->heads == 64 && cfg->hidden % cfg->heads == 0,
               "ac_encoder_create: head_dim must be 64 (hidden=%d heads=%d)", cfg->hidden, cfg->heads);
    AC_REQUIRE(cfg->intermediate % 64 == 0 && cfg->layers > 0 && cfg->max_tokens > 0, "ac_encoder_create: bad dims");
    int rc = ac_device_check();
    if (rc) return rc;
    ac_encoder *e = new ac_encoder();
    e->cfg = *cfg;
    const int H = cfg->hidden, I = cfg->intermediate, L = cfg->layers;
    const size_t T = static_cast<size_t>((cfg->max_tokens + 127) / 128 * 128);
    e->T = T;
#define TRY(x) do { rc = (x); if (rc) { ac_encoder_destroy(e); return rc; } } while (0)
    TRY(pack_f32(e, &e->word, w->word_emb, static_cast<size_t>(cfg->vocab) * H));
    TRY(pack_f32(e, &e->pos, w->pos_emb, static_cast<size_t>(cfg->max_pos) * H));
    TRY(pack_f32(e, &e->type, w->type_emb, static_cast<size_t>(cfg->type_vocab) * H));
    TRY(pack_f32(e, &e->emb_ln_w, w->emb_ln_w, H));
    TRY(pack_f32(e, &e->emb_ln_b, w->emb_ln_b, H));
    e->wqkv_d.assign(L, nullptr); e->wo.assign(L, nullptr); e->w1_d.assign(L, nullptr); e->w2.assign(L, nullptr);
    e->c1qkv.assign(L, nullptr); e->c0qkv.assign(L, nullptr); e->c1f.assign(L, nullptr); e->c0f.assign(L, nullptr);
    e->bo.assign(L, nullptr); e->ln1w.assign(L, nullptr); e->ln1b.assign(L, nullptr);
    e->b2.assign(L, nullptr); e->ln2w.assign(L, nullptr); e->ln2b.assign(L, nullptr);
    const size_t HH = static_cast<size_t>(H) * H;
    for (int l = 0; l < L; ++l) {
        // fused QKV operand [3H, H]: the projection of layer l consumes the sums whose pending LayerNorm is the output
        // LayerNorm of layer l-1 (identity for layer 0: the embeddings arrive normalised)
        TRY(dev_alloc(e, &e->wqkv_d[l], 3 * HH));
        TRY(dev_alloc(e, &e->c1qkv[l], 3 * static_cast<size_t>(H)));
        TRY(dev_alloc(e, &e->c0qkv[l], 3 * static_cast<size_t>(H)));
        const float *ws[3] = {w->q_w[l], w->k_w[l], w->v_w[l]};
        const float *bs[3] = {w->q_b[l], w->k_b[l], w->v_b[l]};
        const float *pg = l ? w->out_ln_w[l - 1] : nullptr, *pb = l ? w->out_ln_b[l - 1] : nullptr;
        for (int j = 0; j < 3; ++j) {
            pack_defer_kernel<<<(H + 7) / 8, 256>>>(ws[j], bs[j], pg, pb, H, H, e->wqkv_d[l] + j * HH, e->c1qkv[l] + j * H,
                                                    e->c0qkv[l] + j * H);
            TRY(check_cuda(cudaGetLastError(), "pack_defer_kernel qkv"));
        }
        TRY(pack_f16(e, &e->wo[l], w->ao_w[l], HH));
        TRY(pack_f32(e, &e->bo[l], w->ao_b[l], H));
        TRY(pack_f32(e, &e->ln1w[l], w->ao_ln_w[l], H));
        TRY(pack_f32(e, &e->ln1b[l], w->ao_ln_b[l], H));
        // FFN1 of layer l consumes the sums pending the attention-output LayerNorm of layer l
        TRY(dev_alloc(e, &e->w1_d[l], static_cast<size_t>(I) * H));
        TRY(dev_alloc(e, &e->c1f[l], I));
        TRY(dev_alloc(e, &e->c0f[l], I));
        pack_defer_kernel<<<(I + 7) / 8, 256>>>(w->ff1_w[l], w->ff1_b[l], w->ao_ln_w[l], w->ao_ln_b[l], I, H, e->w1_d[l], e->c1f[l],
                                                e->c0f[l]);
        TRY(check_cuda(cudaGetLastError(), "pack_defer_kernel ffn1"));
        TRY(pack_f16(e, &e->w2[l], w->ff2_w[l], static_cast<size_t>(H) * I));
        TRY(pack_f32(e, &e->b2[l], w->ff2_b[l], H));
        TRY(pack_f32(e, &e->ln2w[l], w->out_ln_w[l], H));
        TRY(pack_f32(e, &e->ln2b[l], w->out_ln_b[l], H));
    }
    if (cfg->cls_only) {
        TRY(pack_f16(e, &e->w1_last, w->ff1_w[L - 1], static_cast<size_t>(I) * H));
        TRY(pack_f32(e, &e->b1_last, w->ff1_b[L - 1], I));
    }
    TRY(alloc_workspace(e));
    e->p_wqkv_d.resize(L); e->p_wo.resize(L); e->p_w1_d.resize(L); e->p_w2.resize(L);
    for (int l = 0; l < L; ++l) {
        TRY(make_tmap_2d(&e->p_wqkv_d[l], e->wqkv_d[l], 2, 3 * H, H, static_cast<uint64_t>(H) * 2, GEMM2_B_ROWS, 64));
        TRY(make_tmap_2d(&e->p_wo[l], e->wo[l], 2, H, H, static_cast<uint64_t>(H) * 2, GEMM2_B_ROWS, 64));
        TRY(make_tmap_2d(&e->p_w1_d[l], e->w1_d[l], 2, I, H, static_cast<uint64_t>(H) * 2, GEMM2_B_ROWS, 64));
        TRY(make_tmap_2d(&e->p_w2[l], e->w2[l], 2, H, I, static_cast<uint64_t>(I) * 2, GEMM2_B_ROWS, 64));
    }
    if (cfg->cls_only) TRY(make_tmap_2d(&e->p_w1_last, e->w1_last, 2, I, H, static_cast<uint64_t>(H) * 2, GEMM2_B_ROWS, 64));
    TRY(check_cuda(cudaDeviceSynchronize(), "encoder_create sync"));
#undef TRY
    *out = e;
    return AC_OK;
}

// fp32 copy of src, or n zeros when src is NULL (absent biases of ModernBERT's norm_bias / attention_bias / mlp_bias = False)
static int pack_f32_or_zero(ac_encoder *e, float **dst, const float *src, size_t n) {
    if (src) return pack_f32(e, dst, src, n);
    int rc = dev_alloc(e, dst, n);
    if (rc) return rc;
    AC_CUDA(cudaMemset(*dst, 0, n * sizeof(float)));
    return AC_OK;
}

constexpr int ROPE_MAX_POS = 512;

extern "C" int ac_encoder_create_modernbert(const ac_modernbert_config *cfg, const ac_modernbert_weights *w, ac_encoder **out) {
    AC_REQUIRE(cfg && w && out, "ac_encoder_create_modernbert: null argument");
    AC_REQUIRE(cfg->precision == AC_PREC_F16, "ac_encoder_create_modernbert: only AC_PREC_F16 is implemented");
    AC_REQUIRE(cfg->hidden % 128 == 0 && cfg->hidden > 0 && cfg->hidden <= 1024,
               "ac_encoder_create_modernbert: hidden=%d must be a multiple of 128, <= 1024", cfg->hidden);
    AC_REQUIRE(cfg->heads > 0 && cfg->hidden % cfg->heads == 0 && cfg->hidden / cfg->heads == 64,
               "ac_encoder_create_modernbert: head_dim must be 64 (hidden=%d heads=%d)", cfg->hidden, cfg->heads);
    AC_REQUIRE(cfg->intermediate > 0 && cfg->intermediate % 64 == 0,
               "ac_encoder_create_modernbert: intermediate=%d must be a multiple of 64", cfg->intermediate);
    AC_REQUIRE(cfg->layers > 0 && cfg->max_tokens > 0 && cfg->vocab > 0, "ac_encoder_create_modernbert: bad dims");
    AC_REQUIRE(cfg->window && cfg->rope_theta, "ac_encoder_create_modernbert: window and rope_theta arrays are required");
    for (int l = 0; l < cfg->layers; ++l)
        AC_REQUIRE(cfg->window[l] >= 0 && cfg->rope_theta[l] > 0.f, "ac_encoder_create_modernbert: layer %d: window=%d theta=%g",
                   l, cfg->window[l], static_cast<double>(cfg->rope_theta[l]));
    AC_REQUIRE(w->tok_emb && w->emb_norm_w && w->final_norm_w && w->Wqkv && w->Wo && w->mlp_norm_w && w->Wi && w->mlp_Wo &&
                   (cfg->layers == 1 || w->attn_norm_w),
               "ac_encoder_create_modernbert: missing weight");
    int rc = ac_device_check();
    if (rc) return rc;
    ac_encoder *e = new ac_encoder();
    ac_encoder_config &c = e->cfg;
    c.arch = AC_ARCH_MODERNBERT;
    c.layers = cfg->layers; c.hidden = cfg->hidden; c.heads = cfg->heads; c.intermediate = cfg->intermediate;
    c.vocab = cfg->vocab; c.max_pos = ROPE_MAX_POS; c.type_vocab = 1; c.pad_idx = 0;
    c.ln_eps = cfg->norm_eps; c.precision = cfg->precision; c.max_tokens = cfg->max_tokens; c.cls_only = cfg->cls_only;
    const int H = c.hidden, I = c.intermediate, L = c.layers;
    e->T = static_cast<size_t>((cfg->max_tokens + 127) / 128 * 128);
    auto at = [](const float *const *a, int l) -> const float * { return a ? a[l] : nullptr; };
#define TRY(x) do { rc = (x); if (rc) { ac_encoder_destroy(e); return rc; } } while (0)
    TRY(pack_f32(e, &e->word, w->tok_emb, static_cast<size_t>(c.vocab) * H));
    TRY(pack_f32(e, &e->emb_ln_w, w->emb_norm_w, H));
    TRY(pack_f32_or_zero(e, &e->emb_ln_b, w->emb_norm_b, H));
    TRY(pack_f32(e, &e->final_nw, w->final_norm_w, H));
    TRY(pack_f32_or_zero(e, &e->final_nb, w->final_norm_b, H));
    e->wqkv_d.assign(L, nullptr); e->wo.assign(L, nullptr); e->w1_d.assign(L, nullptr); e->w2.assign(L, nullptr);
    e->bqkv.assign(L, nullptr); e->bo.assign(L, nullptr); e->bi.assign(L, nullptr); e->b2.assign(L, nullptr);
    e->attn_nw.assign(L, nullptr); e->attn_nb.assign(L, nullptr); e->mlp_nw.assign(L, nullptr); e->mlp_nb.assign(L, nullptr);
    e->rope.assign(L, nullptr);
    e->window.assign(cfg->window, cfg->window + L);
    const size_t HH = static_cast<size_t>(H) * H;
    std::vector<float2> cs(static_cast<size_t>(ROPE_MAX_POS) * 32);
    for (int l = 0; l < L; ++l) {
        if (l > 0) {
            TRY(pack_f32(e, &e->attn_nw[l], w->attn_norm_w[l], H));
            TRY(pack_f32_or_zero(e, &e->attn_nb[l], at(w->attn_norm_b, l), H));
        }
        TRY(pack_f16(e, &e->wqkv_d[l], w->Wqkv[l], 3 * HH));
        TRY(pack_f32_or_zero(e, &e->bqkv[l], at(w->Wqkv_b, l), 3 * static_cast<size_t>(H)));
        TRY(pack_f16(e, &e->wo[l], w->Wo[l], HH));
        TRY(pack_f32_or_zero(e, &e->bo[l], at(w->Wo_b, l), H));
        TRY(pack_f32(e, &e->mlp_nw[l], w->mlp_norm_w[l], H));
        TRY(pack_f32_or_zero(e, &e->mlp_nb[l], at(w->mlp_norm_b, l), H));
        TRY(dev_alloc(e, &e->w1_d[l], 2 * static_cast<size_t>(I) * H));
        TRY(dev_alloc(e, &e->bi[l], 2 * static_cast<size_t>(I)));
        pack_geglu_kernel<<<(2 * I + 7) / 8, 256>>>(w->Wi[l], at(w->Wi_b, l), I, H, e->w1_d[l], e->bi[l]);
        TRY(check_cuda(cudaGetLastError(), "pack_geglu_kernel"));
        TRY(pack_f16(e, &e->w2[l], w->mlp_Wo[l], static_cast<size_t>(H) * I));
        TRY(pack_f32_or_zero(e, &e->b2[l], at(w->mlp_Wo_b, l), H));
        // RoPE table of this layer's theta, as HF computes it (modeling_modernbert.py:121-154): inv_freq = 1 / theta^(2i/64)
        // and angle = position * inv_freq in fp32, cos / sin of the fp32 angle
        const float theta = cfg->rope_theta[l];
        for (int i = 0; i < 32; ++i) {
            const float inv = 1.0f / powf(theta, static_cast<float>(2 * i) / 64.f);
            for (int pos = 0; pos < ROPE_MAX_POS; ++pos) {
                const float ang = static_cast<float>(pos) * inv;
                cs[static_cast<size_t>(pos) * 32 + i] = make_float2(static_cast<float>(cos(static_cast<double>(ang))),
                                                                    static_cast<float>(sin(static_cast<double>(ang))));
            }
        }
        TRY(dev_alloc(e, &e->rope[l], cs.size()));
        TRY(check_cuda(cudaMemcpy(e->rope[l], cs.data(), cs.size() * sizeof(float2), cudaMemcpyHostToDevice), "rope table"));
    }
    TRY(alloc_workspace(e));
    e->p_wqkv_d.resize(L); e->p_wo.resize(L); e->p_w1_d.resize(L); e->p_w2.resize(L);
    for (int l = 0; l < L; ++l) {
        TRY(make_tmap_2d(&e->p_wqkv_d[l], e->wqkv_d[l], 2, 3 * H, H, static_cast<uint64_t>(H) * 2, GEMM2_B_ROWS, 64));
        TRY(make_tmap_2d(&e->p_wo[l], e->wo[l], 2, H, H, static_cast<uint64_t>(H) * 2, GEMM2_B_ROWS, 64));
        TRY(make_tmap_2d(&e->p_w1_d[l], e->w1_d[l], 2, 2 * I, H, static_cast<uint64_t>(H) * 2, GEMM2_B_ROWS, 64));
        TRY(make_tmap_2d(&e->p_w2[l], e->w2[l], 2, H, I, static_cast<uint64_t>(I) * 2, GEMM2_B_ROWS, 64));
    }
    TRY(check_cuda(cudaDeviceSynchronize(), "encoder_create_modernbert sync"));
#undef TRY
    *out = e;
    return AC_OK;
}

using EpiGelu = EpiLinear<1, true, false>;                  // bias + GELU, fp16 out                       (CLS-only tail)
using EpiResid = EpiLinear<2, false, false>;                // bias + residual, fp32 out (pre-LayerNorm sum, CLS-only tail)
using EpiQKVDefer = EpiLinear<0, true, true, true>;         // r (acc - mu c1) + c0, fp16 out, V third transposed
using EpiGeluDefer16 = EpiLinear<1, true, false, true, 64>; // GELU(r (acc - mu c1) + c0), fp16 out; 16 epilogue warps x 64 columns

// One encoder projection = one CTA-pair GEMM (gemm_tc2.cuh).  tb is the weight's 128-row-box map.  The bias + GELU epilogue of
// FFN1 issues ~17 instructions per element, which two warps per scheduler cannot hide behind a K = 768 mainloop: it runs with
// 16 epilogue warps (measured on a B200: -0.65 ms per 12-layer forward at B*S = 65536, profiles/r02_variants.md).
template <class Epi, int kEpiWarps = GEMM_EPI_WARPS>
static int launch_linear(const CUtensorMap &ta, const CUtensorMap &tb, int M, int N, int K, const Epi &epi, cudaStream_t s) {
    return launch_gemm_tc2<Epi, false, GEMM_KIND_F16, kEpiWarps>(ta, tb, M, N, K, epi, s);
}

// ModernBERT forward (pre-LN): e->x holds the residual stream x (fp32); every LayerNorm is materialised as the fp16 A operand
// of the projection that consumes it, so the projections run on plain fp16 weights with bias epilogues.  (The deferred form
// of the post-LN path folds LN into the consumer as r (acc - mu c1) + c0; on a pre-LN stream, whose row mean grows with
// depth, both that difference and the E[y^2] - mu^2 variance cancel, and the materialised LayerNorm costs one extra
// read of x and fp16 write per half layer.)
static int forward_modernbert(ac_encoder *e, const int32_t *ids, const int32_t *mask, int B, int S, float *out_unit_cls,
                              cudaStream_t s) {
    const ac_encoder_config &c = e->cfg;
    const int H = c.hidden, I = c.intermediate, M = B * S;
    const int S_pad = (S + 7) / 8 * 8;
    const int wpb = 8;
    const int row_blocks = (M + wpb - 1) / wpb;
    int rc;
    // layer 0's attn_norm is the identity: the normalised embeddings are both the stream and the first A operand
    embed_norm_kernel<<<row_blocks, wpb * 32, 0, s>>>(ids, e->word, e->emb_ln_w, e->emb_ln_b, c.ln_eps, M, H, c.vocab, e->x, e->xh);
    AC_LAUNCH_CHECK();
    for (int l = 0; l < c.layers; ++l) {
        if (l > 0) {
            layernorm_kernel<<<row_blocks, wpb * 32, 0, s>>>(e->x, e->attn_nw[l], e->attn_nb[l], c.ln_eps, M, H, nullptr, e->xh);
            AC_LAUNCH_CHECK();
        }
        EpiQKVRope eq{e->bqkv[l], e->qk, e->vT, e->rope[l], M, H, S, S_pad};
        if ((rc = launch_linear(e->m_xh, e->p_wqkv_d[l], M, 3 * H, H, eq, s))) return rc;
        if ((rc = launch_attention(e->m_qk_att, e->m_vt_att, mask, B, S, c.heads, e->ctx, s, e->window[l]))) return rc;
        if (l == c.layers - 1 && c.cls_only && static_cast<size_t>(B) <= e->Bc) {
            // ---- CLS-only tail (classifier.py:1272 pools row 0): Wo + residual, mlp_norm, GeGLU, mlp.Wo + residual and
            // final_norm on the B CLS rows
            const int cb = (B + wpb - 1) / wpb;
            gather_cls_kernel<<<cb, wpb * 32, 0, s>>>(e->ctx, e->x, B, S, H, e->ctx_cls, e->x_cls);
            AC_LAUNCH_CHECK();
            EpiResid eo{e->bo[l], e->x_cls, e->tmp_cls, B, H, H, 0, nullptr, 0, 0, 0, 0};
            if ((rc = launch_linear(e->m_ctx_cls, e->p_wo[l], B, H, H, eo, s))) return rc;
            layernorm_kernel<<<cb, wpb * 32, 0, s>>>(e->tmp_cls, e->mlp_nw[l], e->mlp_nb[l], c.ln_eps, B, H, nullptr, e->xh_cls);
            AC_LAUNCH_CHECK();
            EpiGeGLU eg{e->bi[l], e->ffn_cls, B, 2 * I, I};
            if ((rc = launch_linear(e->m_xh_cls, e->p_w1_d[l], B, 2 * I, H, eg, s))) return rc;
            EpiResid e2{e->b2[l], e->tmp_cls, e->x_cls, B, H, H, 0, nullptr, 0, 0, 0, 0};
            if ((rc = launch_linear(e->m_ffn_cls, e->p_w2[l], B, H, I, e2, s))) return rc;
            layernorm_kernel<<<cb, wpb * 32, 0, s>>>(e->x_cls, e->final_nw, e->final_nb, c.ln_eps, B, H, e->tmp_cls, nullptr);
            AC_LAUNCH_CHECK();
            if ((rc = launch_cls_normalize(e->tmp_cls, B, 1, H, out_unit_cls, s))) return rc;
            e->last_B = B;
            e->last_S = S;
            e->last_cls_only = true;
            return AC_OK;
        }
        // x' = x + Wo(ctx) into e->tmp, then x = x' + mlp.Wo(GeGLU(Wi(mlp_norm(x')))) back into e->x
        EpiResid eo{e->bo[l], e->x, e->tmp, M, H, H, 0, nullptr, 0, 0, 0, 0};
        if ((rc = launch_linear(e->m_ctx, e->p_wo[l], M, H, H, eo, s))) return rc;
        layernorm_kernel<<<row_blocks, wpb * 32, 0, s>>>(e->tmp, e->mlp_nw[l], e->mlp_nb[l], c.ln_eps, M, H, nullptr, e->xh);
        AC_LAUNCH_CHECK();
        EpiGeGLU eg{e->bi[l], e->ffn, M, 2 * I, I};
        if ((rc = launch_linear(e->m_xh, e->p_w1_d[l], M, 2 * I, H, eg, s))) return rc;
        EpiResid e2{e->b2[l], e->tmp, e->x, M, H, H, 0, nullptr, 0, 0, 0, 0};
        if ((rc = launch_linear(e->m_ffn, e->p_w2[l], M, H, I, e2, s))) return rc;
    }
    // full hidden state (cls_only = 0): final_norm on every row
    layernorm_kernel<<<row_blocks, wpb * 32, 0, s>>>(e->x, e->final_nw, e->final_nb, c.ln_eps, M, H, e->tmp, nullptr);
    AC_LAUNCH_CHECK();
    if ((rc = launch_cls_normalize(e->tmp, B, S, H, out_unit_cls, s))) return rc;
    e->last_B = B;
    e->last_S = S;
    e->last_cls_only = false;
    e->last_hidden = e->tmp;
    return AC_OK;
}

extern "C" int ac_encoder_forward_cls(ac_encoder *e, const int32_t *ids, const int32_t *mask, const int32_t *type_ids,
                                      int B, int S, float *out_unit_cls, ac_stream_t stream) {
    AC_REQUIRE(e && ids && out_unit_cls, "ac_encoder_forward_cls: null argument");
    AC_REQUIRE(B > 0 && S > 0, "ac_encoder_forward_cls: B=%d S=%d", B, S);
    if (S > 512) {
        set_error("ac_encoder_forward_cls: S=%d > 512 is not supported (the reference truncates at max_length = 512)", S);
        return AC_E_UNSUPPORTED;
    }
    AC_REQUIRE(static_cast<int64_t>(B) * S <= e->cfg.max_tokens, "ac_encoder_forward_cls: B*S=%lld exceeds max_tokens=%d",
               static_cast<long long>(B) * S, e->cfg.max_tokens);
    AC_REQUIRE(S <= e->cfg.max_pos, "ac_encoder_forward_cls: S exceeds max_position_embeddings");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const ac_encoder_config &c = e->cfg;
    const int H = c.hidden, I = c.intermediate, M = B * S;
    const int S_pad = (S + 7) / 8 * 8;
    AC_REQUIRE(static_cast<size_t>(B) * H * S_pad <= e->vt_elems,
               "ac_encoder_forward_cls: B=%d sequences of S=%d exceed the transposed-V workspace; split the batch", B, S);
    int rc;
    if (e->vt_B != B || e->vt_S != S) {
        // V^T view of this call: rows (b, h, d), S_pad keys per row; box = 64 keys x 64 head dims
        if ((rc = make_tmap_2d(&e->m_vt_att, e->vT, 2, static_cast<uint64_t>(B) * H, S_pad, static_cast<uint64_t>(S_pad) * 2, 64, 64)))
            return rc;
        e->vt_B = B; e->vt_S = S;
    }
    if (c.arch == AC_ARCH_MODERNBERT) return forward_modernbert(e, ids, mask, B, S, out_unit_cls, s);
    const int wpb = 8;
    const int row_blocks = (M + wpb - 1) / wpb;
    const int nparts = H / 128;
    const int64_t pstride = static_cast<int64_t>(e->T);

    // e->x holds the un-normalised residual sums y, e->xh their fp16 copy; the LayerNorm still pending on y is carried as
    // (gamma, beta, row statistics).  The embeddings arrive normalised: identity LayerNorm pending.
    embed_ln_kernel<<<row_blocks, wpb * 32, 0, s>>>(ids, type_ids, e->word, e->pos, e->type, e->emb_ln_w, e->emb_ln_b,
                                                    c.ln_eps, B, S, H, c.arch, c.pad_idx, c.vocab, c.max_pos,
                                                    c.type_vocab, e->x, e->xh);
    AC_LAUNCH_CHECK();
    const float *pg = e->ones, *pb = e->zeros;
    const float2 *st_in = e->stats_id;
    for (int l = 0; l < c.layers; ++l) {
        EpiQKVDefer eq{e->c0qkv[l], nullptr, e->qk, M, 3 * H, 2 * H, 0, e->vT, 2 * H, S, S_pad, H, e->c1qkv[l], st_in};
        if ((rc = launch_linear(e->m_xh, e->p_wqkv_d[l], M, 3 * H, H, eq, s))) return rc;
        if ((rc = launch_attention(e->m_qk_att, e->m_vt_att, mask, B, S, c.heads, e->ctx, s))) return rc;
        if (l == c.layers - 1 && c.cls_only && static_cast<size_t>(B) <= e->Bc) {
            // ---- CLS-only tail of the last layer (classifier.py:1272 pools row 0): M = B rows.  LN_pending is materialised on
            // the CLS rows and the tail runs on ordinary LayerNorm kernels and the plain (not gamma-scaled) FFN1 weight
            const int cb = (B + wpb - 1) / wpb;
            if (l == 0)   // single-layer encoder: nothing is pending on the (already normalised) embeddings
                gather_cls_kernel<<<cb, wpb * 32, 0, s>>>(e->ctx, e->x, B, S, H, e->ctx_cls, e->x_cls);
            else
                gather_cls_ln_kernel<<<cb, wpb * 32, 0, s>>>(e->ctx, e->x, B, S, H, pg, pb, c.ln_eps, e->ctx_cls, e->x_cls);
            AC_LAUNCH_CHECK();
            EpiResid eo{e->bo[l], e->x_cls, e->tmp_cls, B, H, H, 0, nullptr, 0, 0, 0, 0};
            if ((rc = launch_linear(e->m_ctx_cls, e->p_wo[l], B, H, H, eo, s))) return rc;
            layernorm_kernel<<<cb, wpb * 32, 0, s>>>(e->tmp_cls, e->ln1w[l], e->ln1b[l], c.ln_eps, B, H, e->x_cls, e->xh_cls);
            AC_LAUNCH_CHECK();
            EpiGelu e1{e->b1_last, nullptr, e->ffn_cls, B, I, I, 0, nullptr, 0, 0, 0, 0};
            if ((rc = launch_linear(e->m_xh_cls, e->p_w1_last, B, I, H, e1, s))) return rc;
            EpiResid e2{e->b2[l], e->x_cls, e->tmp_cls, B, H, H, 0, nullptr, 0, 0, 0, 0};
            if ((rc = launch_linear(e->m_ffn_cls, e->p_w2[l], B, H, I, e2, s))) return rc;
            layernorm_kernel<<<cb, wpb * 32, 0, s>>>(e->tmp_cls, e->ln2w[l], e->ln2b[l], c.ln_eps, B, H, e->x_cls, nullptr);
            AC_LAUNCH_CHECK();
            if ((rc = launch_cls_normalize(e->x_cls, B, 1, H, out_unit_cls, s))) return rc;
            e->last_B = B;
            e->last_S = S;
            e->last_cls_only = true;
            return AC_OK;
        }
        // attention output projection + residual: y <- ctx Wo^T + bo + LN_pending(y); statistics of the new sums
        EpiResidDefer eo{e->bo[l], e->x, e->xh, st_in, pg, pb, e->parts, pstride, M, H, H};
        if ((rc = launch_linear(e->m_ctx, e->p_wo[l], M, H, H, eo, s))) return rc;
        ln_stats_kernel<<<(M + 255) / 256, 256, 0, s>>>(e->parts, nparts, pstride, M, H, c.ln_eps, e->stats_b);
        AC_LAUNCH_CHECK();
        EpiGeluDefer16 e1{e->c0f[l], nullptr, e->ffn, M, I, I, 0, nullptr, 0, 0, 0, 0, e->c1f[l], e->stats_b};
        if ((rc = launch_linear<EpiGeluDefer16, 16>(e->m_xh, e->p_w1_d[l], M, I, H, e1, s))) return rc;
        // FFN output projection + residual: y <- ffn W2^T + b2 + LN_attention_output(y)
        EpiResidDefer e2{e->b2[l], e->x, e->xh, e->stats_b, e->ln1w[l], e->ln1b[l], e->parts, pstride, M, H, H};
        if ((rc = launch_linear(e->m_ffn, e->p_w2[l], M, H, I, e2, s))) return rc;
        ln_stats_kernel<<<(M + 255) / 256, 256, 0, s>>>(e->parts, nparts, pstride, M, H, c.ln_eps, e->stats_a);
        AC_LAUNCH_CHECK();
        pg = e->ln2w[l];
        pb = e->ln2b[l];
        st_in = e->stats_a;
    }
    // full hidden state requested (cls_only = 0): materialise the last LayerNorm for every row
    layernorm_kernel<<<row_blocks, wpb * 32, 0, s>>>(e->x, pg, pb, c.ln_eps, M, H, e->tmp, nullptr);
    AC_LAUNCH_CHECK();
    if ((rc = launch_cls_normalize(e->tmp, B, S, H, out_unit_cls, s))) return rc;
    e->last_B = B;
    e->last_S = S;
    e->last_cls_only = false;
    e->last_hidden = e->tmp;
    return AC_OK;
}

extern "C" int ac_encoder_last_hidden(ac_encoder *e, float *out, int64_t n_floats, ac_stream_t stream) {
    AC_REQUIRE(e && out, "ac_encoder_last_hidden: null argument");
    AC_REQUIRE(!e->last_cls_only, "ac_encoder_last_hidden: the previous forward computed only the CLS rows of the last layer "
                                  "(create the encoder with cls_only = 0 to keep the full hidden state)");
    const int64_t have = static_cast<int64_t>(e->last_B) * e->last_S * e->cfg.hidden;
    AC_REQUIRE(n_floats <= have, "ac_encoder_last_hidden: asked %lld floats, have %lld", (long long)n_floats, (long long)have);
    AC_CUDA(cudaMemcpyAsync(out, e->last_hidden ? e->last_hidden : e->x, n_floats * sizeof(float), cudaMemcpyDeviceToDevice,
                            static_cast<cudaStream_t>(stream)));
    return AC_OK;
}

// the encoder's attention exposed for parity tests: the tensor maps the encoder caches, built over caller buffers, and the
// encoder's own dispatch
extern "C" int ac_attention(const void *qk, int64_t qk_rows, const void *vT, const int32_t *mask, int B, int S, int heads,
                            int window, void *ctx, ac_stream_t stream) {
    AC_REQUIRE(qk && vT && ctx, "ac_attention: null argument");
    AC_REQUIRE(B > 0 && S > 0 && S <= 512 && heads > 0 && window >= 0, "ac_attention: B=%d S=%d heads=%d window=%d", B, S, heads,
               window);
    AC_REQUIRE(qk_rows >= static_cast<int64_t>(B) * S, "ac_attention: qk has %lld rows, B*S = %lld", (long long)qk_rows,
               static_cast<long long>(B) * S);
    int rc = ac_device_check();
    if (rc) return rc;
    const int H = heads * 64, S_pad = (S + 7) / 8 * 8;
    CUtensorMap tqk, tvt;
    if ((rc = make_tmap_2d(&tqk, qk, 2, static_cast<uint64_t>(qk_rows), 2 * H, static_cast<uint64_t>(2 * H) * 2, 128, 64))) return rc;
    if ((rc = make_tmap_2d(&tvt, vT, 2, static_cast<uint64_t>(B) * H, S_pad, static_cast<uint64_t>(S_pad) * 2, 64, 64))) return rc;
    return launch_attention(tqk, tvt, mask, B, S, heads, static_cast<__half *>(ctx), static_cast<cudaStream_t>(stream), window);
}

// generic tensor-core linear exposed for parity tests / roofline measurement (the encoder's CTA-pair GEMM with a plain epilogue).
//   precision AC_PREC_TF32: X, W fp32 (used as stored, tf32 truncation by the MMA unless pre-rounded), Y fp32
//   precision AC_PREC_F16 : X, W fp16, Y fp32 (out_half = 0) or fp16 (out_half = 1)
template <int MODE, bool OUT_HALF, int KIND>
static int linear_tc_dispatch(const CUtensorMap &ta, const CUtensorMap &tb, const float *bias, const float *residual, void *Y,
                              int M, int N, int K, int round_out, cudaStream_t s) {
    EpiLinear<MODE, OUT_HALF, false> e{bias, residual, Y, M, N, N, round_out, nullptr, 0, 0, 0, 0};
    return launch_gemm_tc2<EpiLinear<MODE, OUT_HALF, false>, false, KIND>(ta, tb, M, N, K, e, s);
}

extern "C" int ac_linear_tc(const void *X, const void *W, const float *bias, const float *residual, void *Y, int M, int N,
                            int K, int epi, int round_out, int precision, int out_half, ac_stream_t stream) {
    AC_REQUIRE(X && W && Y && bias && M > 0 && N > 0 && K > 0, "ac_linear_tc: bad arguments (bias is required)");
    AC_REQUIRE(epi >= 0 && epi <= 2 && (epi != 2 || residual), "ac_linear_tc: bad epilogue");
    AC_REQUIRE(precision == AC_PREC_TF32 || precision == AC_PREC_F16, "ac_linear_tc: bad precision");
    AC_REQUIRE(!(out_half && epi == 2), "ac_linear_tc: the residual epilogue writes fp32");
    const int es = precision == AC_PREC_F16 ? 2 : 4;
    AC_REQUIRE((K * es) % 16 == 0 && N % 8 == 0, "ac_linear_tc: rows must be 16-byte multiples and N %% 8 == 0");
    int rc = ac_device_check();
    if (rc) return rc;
    CUtensorMap ta, tb;
    const uint32_t bk = 128 / es;
    if ((rc = make_tmap_2d(&ta, X, es, M, K, static_cast<uint64_t>(K) * es, GEMM_BLOCK_M, bk))) return rc;
    if ((rc = make_tmap_2d(&tb, W, es, N, K, static_cast<uint64_t>(K) * es, GEMM2_B_ROWS, bk))) return rc;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (precision == AC_PREC_TF32) {
        AC_REQUIRE(!out_half, "ac_linear_tc: tf32 path writes fp32");
        if (epi == 0) return linear_tc_dispatch<0, false, GEMM_KIND_TF32>(ta, tb, bias, residual, Y, M, N, K, round_out, s);
        if (epi == 1) return linear_tc_dispatch<1, false, GEMM_KIND_TF32>(ta, tb, bias, residual, Y, M, N, K, round_out, s);
        return linear_tc_dispatch<2, false, GEMM_KIND_TF32>(ta, tb, bias, residual, Y, M, N, K, round_out, s);
    }
    if (out_half) {
        if (epi == 0) return linear_tc_dispatch<0, true, GEMM_KIND_F16>(ta, tb, bias, residual, Y, M, N, K, 0, s);
        return linear_tc_dispatch<1, true, GEMM_KIND_F16>(ta, tb, bias, residual, Y, M, N, K, 0, s);
    }
    if (epi == 0) return linear_tc_dispatch<0, false, GEMM_KIND_F16>(ta, tb, bias, residual, Y, M, N, K, 0, s);
    if (epi == 1) return linear_tc_dispatch<1, false, GEMM_KIND_F16>(ta, tb, bias, residual, Y, M, N, K, 0, s);
    return linear_tc_dispatch<2, false, GEMM_KIND_F16>(ta, tb, bias, residual, Y, M, N, K, 0, s);
}
