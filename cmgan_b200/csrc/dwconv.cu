// GLU + depthwise Conv1d(k = 31, zero pad 15/15, bias) of the conformer convolution module.
// Reference: conformer.py:30-48,164-168.  Input g (M, 256) = pointwise-conv output, u = g[:, :128] * sigmoid(g[:, 128:]),
// out[tok, c] = bias[c] + sum_k w[c, k] * u[tok + k - 15, c] along the sequence axis (strided rows, SeqGeom).
//
// HBM-bound streaming kernels.  The (sequence, 16-token tile) space is flattened and cut into equal contiguous ranges, one per resident
// block (persistent grid, no tail wave).  A block walks its range with a 64-row ring of staged rows in shared memory: every row of g
// (and of dz) is read from global memory once and its sigmoid evaluated once -- no halo re-staging -- and the rows of tile k + 2 are
// fetched into registers before tile k is computed, so the global-load latency hides under the FMA sweep.  Thread = (channel, 8-token
// half of the tile); the taps (and the tap gradients) live in registers.
#include "common.cuh"
#include "../../include/cmgan_b200.h"

namespace {

constexpr int CH = 128, KS = 31, PADL = 15, C4 = CH / 4;
constexpr int CK = 16;                 // rows per chunk = tokens per tile
constexpr int RING = 64;               // ring rows: chunks k - 1, k, k + 1 are read while chunk k + 2 is written
constexpr int TOK = 8;                 // tokens per thread per tile
constexpr int SWEEP = TOK + KS - 1;    // 38 staged rows feed 8 consecutive tokens

struct ChunkRegs {
    float4 a[2], b[2], z[2];
};

// rows of chunk ch (tokens 16 ch .. 16 ch + 15) -> registers; rows outside the sequence read as zeros
template <bool BWD>
__device__ __forceinline__ void load_chunk(ChunkRegs& r, const float* __restrict__ g, const float* __restrict__ dz, long base, long tok_stride,
                                           int ch, int L) {
#pragma unroll
    for (int j = 0; j < 2; ++j) {
        const int idx = threadIdx.x + 256 * j, row = idx >> 5, c4 = idx & 31;
        const int tok = ch * CK + row;
        r.a[j] = r.b[j] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (BWD) r.z[j] = r.a[j];
        if (tok >= 0 && tok < L) {
            const long grow = base + (long)tok * tok_stride;
            const float4* p = reinterpret_cast<const float4*>(g + grow * (2 * CH));
            r.a[j] = __ldg(p + c4);
            r.b[j] = __ldg(p + C4 + c4);
            if (BWD) r.z[j] = __ldg(reinterpret_cast<const float4*>(dz + grow * CH) + c4);
        }
    }
}

template <bool BWD>
__device__ __forceinline__ void store_chunk(const ChunkRegs& r, float* U, float* SG, float* DZ, int ch) {
#pragma unroll
    for (int j = 0; j < 2; ++j) {
        const int idx = threadIdx.x + 256 * j, row = idx >> 5, c4 = idx & 31;
        const int rr = (ch * CK + row) & (RING - 1);
        const float4 a = r.a[j], b = r.b[j];
        const float4 s = make_float4(sigmoidf_(b.x), sigmoidf_(b.y), sigmoidf_(b.z), sigmoidf_(b.w));
        reinterpret_cast<float4*>(U)[rr * C4 + c4] = make_float4(a.x * s.x, a.y * s.y, a.z * s.z, a.w * s.w);
        if (BWD) {
            reinterpret_cast<float4*>(SG)[rr * C4 + c4] = s;
            reinterpret_cast<float4*>(DZ)[rr * C4 + c4] = r.z[j];
        }
    }
}

// Ragged batch (common.cuh): the (sequence, tile) space holds the valid sequences only, each with its own tile count -- batch item b
// contributes nseq_b sequences of tps_b tiles (time axis: F sequences of frames[b] tokens; frequency axis: frames[b] sequences of F
// tokens).  A flat tile index is mapped back by a walk over the batch items (B is small; one walk per contiguous run of a block).
__device__ __forceinline__ long varlen_items(const SeqGeom& sg, const int* __restrict__ frames, int axis, int b, int& L, int& tps) {
    const int n = varlen_frames(frames, b, axis == 0 ? sg.L : sg.n_inner);
    L = axis == 0 ? n : sg.L;
    tps = (L + CK - 1) / CK;
    return (long)(axis == 0 ? sg.n_inner : n) * tps;
}
__device__ long varlen_total(const SeqGeom& sg, const int* __restrict__ frames, int axis) {
    long total = 0;
    int L, tps;
    for (int b = 0; b < sg.n_seq / sg.n_inner; ++b) total += varlen_items(sg, frames, axis, b, L, tps);
    return total;
}
// flat tile index (< varlen_total) -> sequence s, tile k within it, tiles / tokens of that sequence
__device__ __forceinline__ void varlen_tile(const SeqGeom& sg, const int* __restrict__ frames, int axis, long tile, int& s, int& k, int& tps, int& L) {
    int b = 0;
    for (long cnt; tile >= (cnt = varlen_items(sg, frames, axis, b, L, tps)); ++b) tile -= cnt;
    s = b * sg.n_inner + (int)(tile / tps);
    k = (int)(tile % tps);
}

// forward.  bn_sums (optional): per-channel sum / sum of squares of the output (sums[c * 2 + {0, 1}], BatchNorm1d batch statistics,
// conformer.py:169) accumulated here instead of by a separate pass over `out`.  VAR: ragged batch (frames, axis), see varlen_tile.
template <bool VAR>
__global__ void __launch_bounds__(256, 3) glu_dwconv_fwd_kernel(const float* __restrict__ g, SeqGeom sg, const float* __restrict__ w,
                                                                const float* __restrict__ bias, float* __restrict__ out,
                                                                double* __restrict__ bn_sums, const int* __restrict__ frames, int axis) {
    __shared__ __align__(16) float U[RING * CH];
    const int c = threadIdx.x & (CH - 1), half = threadIdx.x >> 7;
    float wr[KS];
#pragma unroll
    for (int k = 0; k < KS; ++k) wr[k] = __ldg(w + c * KS + k);
    const float bs = __ldg(bias + c);
    float s1 = 0.f, s2 = 0.f;
    const int tps_u = (sg.L + CK - 1) / CK;
    const long total = VAR ? varlen_total(sg, frames, axis) : (long)sg.n_seq * tps_u;
    long tile = total * blockIdx.x / gridDim.x;
    const long hi = total * (blockIdx.x + 1) / gridDim.x;
    ChunkRegs regs;
    while (tile < hi) {
        int s, k0, tps = tps_u, L = sg.L;
        if (VAR) {
            varlen_tile(sg, frames, axis, tile, s, k0, tps, L);
        } else {
            s = (int)(tile / tps); k0 = (int)(tile % tps);
        }
        const int kend = (int)min((long)tps, k0 + (hi - tile));
        const long base = seq_base(sg, s);
        __syncthreads();                                        // the previous run is done with the ring
#pragma unroll 1
        for (int ch = k0 - 1; ch <= k0 + 1; ++ch) {
            load_chunk<false>(regs, g, nullptr, base, sg.tok_stride, ch, L);
            store_chunk<false>(regs, U, nullptr, nullptr, ch);
        }
        __syncthreads();
#pragma unroll 1
        for (int k = k0; k < kend; ++k) {
            load_chunk<false>(regs, g, nullptr, base, sg.tok_stride, k + 2, L);
            const int tok0 = k * CK + half * TOK;
            const int rs = (tok0 - PADL) & (RING - 1), wm = RING - rs;          // sweep row m lives at ring row (rs + m) mod 64
            const float* p1 = U + rs * CH + c;
            const float* p2 = p1 - RING * CH;
            float acc[TOK];
#pragma unroll
            for (int i = 0; i < TOK; ++i) acc[i] = bs;
#pragma unroll
            for (int m = 0; m < SWEEP; ++m) {
                const float u = (m < wm ? p1 : p2)[m * CH];
#pragma unroll
                for (int i = 0; i < TOK; ++i)
                    if (m - i >= 0 && m - i < KS) acc[i] = fmaf(wr[m - i], u, acc[i]);
            }
#pragma unroll
            for (int i = 0; i < TOK; ++i) {
                const int tok = tok0 + i;
                if (tok < L) {
                    out[(base + (long)tok * sg.tok_stride) * CH + c] = acc[i];
                    s1 += acc[i];
                    s2 = fmaf(acc[i], acc[i], s2);
                }
            }
            store_chunk<false>(regs, U, nullptr, nullptr, k + 2);
            __syncthreads();
        }
        tile += kend - k0;
    }
    if (bn_sums) {
        __syncthreads();
        if (half) { U[c] = s1; U[CH + c] = s2; }
        __syncthreads();
        if (!half) {
            atomicAdd(bn_sums + c * 2, (double)s1 + (double)U[c]);
            atomicAdd(bn_sums + c * 2 + 1, (double)s2 + (double)U[CH + c]);
        }
    }
}

// backward.  dz = grad wrt out (M, 128).  dg (M, 256) overwritten; dw (128, 31), dbias (128) accumulated.
//   du[tok]  = sum_k w[k] dz[tok - k + 15]          dg_a = du sigmoid(b),  dg_b = du u (1 - sigmoid(b))
//   dw[k]   += dz[tok] u[tok + k - 15]              dbias += dz[tok]
__global__ void __launch_bounds__(256, 2) glu_dwconv_bwd_kernel(const float* __restrict__ g, const float* __restrict__ dz, SeqGeom sg,
                                                                const float* __restrict__ w, float* __restrict__ dg, float* __restrict__ dw,
                                                                float* __restrict__ dbias, int rnd) {
    extern __shared__ __align__(16) float smem[];
    float* U = smem;                    // [RING][CH]
    float* DZ = U + RING * CH;
    float* SG = DZ + RING * CH;
    const int c = threadIdx.x & (CH - 1), half = threadIdx.x >> 7;
    float wr[KS], dwr[KS];
#pragma unroll
    for (int k = 0; k < KS; ++k) { wr[k] = __ldg(w + c * KS + k); dwr[k] = 0.f; }
    float db = 0.f;
    const int tps = (sg.L + CK - 1) / CK;
    const long total = (long)sg.n_seq * tps;
    long tile = total * blockIdx.x / gridDim.x;
    const long hi = total * (blockIdx.x + 1) / gridDim.x;
    ChunkRegs regs;
    while (tile < hi) {
        const int s = (int)(tile / tps), k0 = (int)(tile % tps);
        const int kend = (int)min((long)tps, k0 + (hi - tile));
        const long base = seq_base(sg, s);
        __syncthreads();
#pragma unroll 1
        for (int ch = k0 - 1; ch <= k0 + 1; ++ch) {
            load_chunk<true>(regs, g, dz, base, sg.tok_stride, ch, sg.L);
            store_chunk<true>(regs, U, SG, DZ, ch);
        }
        __syncthreads();
#pragma unroll 1
        for (int k = k0; k < kend; ++k) {
            load_chunk<true>(regs, g, dz, base, sg.tok_stride, k + 2, sg.L);
            const int tok0 = k * CK + half * TOK;
            const int rs = (tok0 - PADL) & (RING - 1), wm = RING - rs;
            const int off1 = rs * CH + c, off2 = off1 - RING * CH;
            float du[TOK], dzc[TOK];
#pragma unroll
            for (int i = 0; i < TOK; ++i) du[i] = 0.f;
            // staged row m = token tok0 - 15 + m: feeds du of token i with tap k = 30 - m + i
#pragma unroll
            for (int m = 0; m < SWEEP; ++m) {
                const float z = DZ[(m < wm ? off1 : off2) + m * CH];
                if (m >= PADL && m < PADL + TOK) dzc[m - PADL] = z;
#pragma unroll
                for (int i = 0; i < TOK; ++i)
                    if (m - i >= 0 && m - i < KS) du[i] = fmaf(wr[KS - 1 - m + i], z, du[i]);
            }
#pragma unroll
            for (int i = 0; i < TOK; ++i) db += dzc[i];
            // dw[k] += dz[token i] * u[row m],  k = m - i
#pragma unroll
            for (int m = 0; m < SWEEP; ++m) {
                const float u = U[(m < wm ? off1 : off2) + m * CH];
#pragma unroll
                for (int i = 0; i < TOK; ++i)
                    if (m - i >= 0 && m - i < KS) dwr[m - i] = fmaf(dzc[i], u, dwr[m - i]);
            }
#pragma unroll
            for (int i = 0; i < TOK; ++i) {
                const int tok = tok0 + i;
                if (tok < sg.L) {
                    const int rr = (tok & (RING - 1)) * CH + c;
                    const float sg_ = SG[rr], u = U[rr];
                    float* o = dg + (base + (long)tok * sg.tok_stride) * (2 * CH) + c;
                    o[0] = cmgan_maybe_rna(du[i] * sg_, rnd);                    // dg feeds two tensor-core contractions
                    o[CH] = cmgan_maybe_rna(du[i] * u * (1.f - sg_), rnd);
                }
            }
            store_chunk<true>(regs, U, SG, DZ, k + 2);
            __syncthreads();
        }
        tile += kend - k0;
    }
    // the two token halves of a channel are combined in shared memory: one atomic per (block, channel, tap)
    __syncthreads();
    if (half) {
#pragma unroll
        for (int k = 0; k < KS; ++k) U[k * CH + c] = dwr[k];
        U[KS * CH + c] = db;
    }
    __syncthreads();
    if (!half) {
#pragma unroll
        for (int k = 0; k < KS; ++k) atomicAdd(dw + c * KS + k, dwr[k] + U[k * CH + c]);
        atomicAdd(dbias + c, db + U[KS * CH + c]);
    }
}

int resident_grid(long total, int per_sm) {
    const long slots = 148L * per_sm;
    return (int)(total < slots ? total : slots);
}

}  // namespace

static int glu_dwconv_fwd_launch(const float* g, const float* w, const float* bias, int B, int T, int F, int axis, const int* frames, float* out,
                                 double* bn_sums, void* stream) {
    CMGAN_REQUIRE(g && w && bias && out && (((uintptr_t)g) & 15) == 0, "cmgan_glu_dwconv_fwd: bad pointer");
    CMGAN_REQUIRE(axis == 0 || axis == 1, "cmgan_glu_dwconv_fwd: bad axis");
    SeqGeom sg = make_seq_geom(B, T, F, axis);
    if (sg.n_seq == 0 || sg.L == 0) return 0;
    const long total = (long)sg.n_seq * cdiv(sg.L, CK);      // a ragged batch has at most this many tiles
    if (frames) glu_dwconv_fwd_kernel<true><<<resident_grid(total, 3), 256, 0, (cudaStream_t)stream>>>(g, sg, w, bias, out, nullptr, frames, axis);
    else glu_dwconv_fwd_kernel<false><<<resident_grid(total, 3), 256, 0, (cudaStream_t)stream>>>(g, sg, w, bias, out, bn_sums, nullptr, axis);
    return cmgan_check_launch("glu_dwconv_fwd_kernel");
}

CMGAN_API int cmgan_glu_dwconv_fwd(const float* g, const float* w, const float* bias, int B, int T, int F, int axis, float* out,
                                   double* bn_sums, void* stream) {
    return glu_dwconv_fwd_launch(g, w, bias, B, T, F, axis, nullptr, out, bn_sums, stream);
}

// ragged batch (frames: device int[B], 1 <= frames[b] <= T); inference only (no BatchNorm batch statistics).  Rows of padded frames are
// neither read nor written, and the persistent partition spans the valid tiles only.
CMGAN_API int cmgan_glu_dwconv_fwd_varlen(const float* g, const float* w, const float* bias, int B, int T, int F, int axis, const int* frames,
                                          float* out, void* stream) {
    CMGAN_REQUIRE(frames, "cmgan_glu_dwconv_fwd_varlen: null frames");
    return glu_dwconv_fwd_launch(g, w, bias, B, T, F, axis, frames, out, nullptr, stream);
}

CMGAN_API int cmgan_glu_dwconv_bwd(const float* g, const float* dz, const float* w, int B, int T, int F, int axis, float* dg, float* dw,
                                   float* dbias, void* stream) {
    CMGAN_REQUIRE(g && dz && w && dg && dw && dbias && ((((uintptr_t)g) | ((uintptr_t)dz)) & 15) == 0, "cmgan_glu_dwconv_bwd: bad pointer");
    CMGAN_REQUIRE(axis == 0 || axis == 1, "cmgan_glu_dwconv_bwd: bad axis");
    SeqGeom sg = make_seq_geom(B, T, F, axis);
    if (sg.n_seq == 0 || sg.L == 0) return 0;
    static bool attr_set = false;
    const int smem = 3 * RING * CH * (int)sizeof(float);
    if (!attr_set) {
        cudaError_t e = cudaFuncSetAttribute(glu_dwconv_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        CMGAN_REQUIRE(e == cudaSuccess, "cmgan_glu_dwconv_bwd: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
        attr_set = true;
    }
    const long total = (long)sg.n_seq * cdiv(sg.L, CK);
    glu_dwconv_bwd_kernel<<<resident_grid(total, 2), 256, smem, (cudaStream_t)stream>>>(g, dz, sg, w, dg, dw, dbias, g_cmgan_round_tf32);
    return cmgan_check_launch("glu_dwconv_bwd_kernel");
}
