// Multi-head self-attention with Shaw relative positions, flash style (no (L, L) tensors in HBM).
// Reference: conformer.py:100-131.  scores[i, j] = 0.25 * q_i . (k_j + E[clamp(i - j, +-512) + 512]),
// softmax over j, out_i = sum_j p_ij v_j; 4 heads x 16, E (1025, 16) shared by the heads.
//
// Layout: qkv rows (M, 192) = [q (h d) | k (h d) | v (h d)] channel-last; a sequence is a strided set of
// rows (SeqGeom: time axis or frequency axis of the (B, T, F) grid), so no transposes are ever made.
// One thread owns one query (forward, dq), one key (dk/dv) or one relative distance (dE); the operand
// that is shared by the whole block is read from shared memory as a broadcast, the per-thread operand
// from a window padded to 20 floats per row (conflict-free 128-bit reads).
#include "common.cuh"
#include "../../include/cmgan_b200.h"

namespace {

constexpr int D = 16, H = 4, CQ = 64, LDQ = 192;
constexpr int NTH = 128;     // threads per block = queries (or keys / distances) per block
constexpr int TILE = 64;     // rows of the broadcast operand staged per step
constexpr int WROWS = NTH + TILE - 1;
constexpr int WLD = 20;
constexpr int MAXPOS = 512;
constexpr float SCALE_LOG2E = 0.25f * 1.4426950408889634f;
constexpr float LN2 = 0.6931471805599453f;

__device__ __forceinline__ void ld16(const float* p, float v[D]) {
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        float4 t = *reinterpret_cast<const float4*>(p + 4 * q);
        v[4 * q] = t.x; v[4 * q + 1] = t.y; v[4 * q + 2] = t.z; v[4 * q + 3] = t.w;
    }
}
__device__ __forceinline__ void st16(float* p, const float v[D]) {
#pragma unroll
    for (int q = 0; q < 4; ++q) *reinterpret_cast<float4*>(p + 4 * q) = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
}
__device__ __forceinline__ int clampi(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }

// stage `n` rows (16 floats each) of a strided qkv column block into dense smem rows of stride 16
__device__ __forceinline__ void stage_rows16(float* dst, const float* src_base, long row0_off, long tok_stride, int first, int n,
                                             int L, float mul) {
    for (int idx = threadIdx.x; idx < n * 4; idx += NTH) {
        int r = idx >> 2, q4 = idx & 3;
        int tok = first + r;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (tok >= 0 && tok < L) v = __ldg(reinterpret_cast<const float4*>(src_base + (row0_off + (long)tok * tok_stride) * LDQ) + q4);
        v.x *= mul; v.y *= mul; v.z *= mul; v.w *= mul;
        *reinterpret_cast<float4*>(dst + r * D + q4 * 4) = v;
    }
}
// same but into the padded (WLD) window layout
__device__ __forceinline__ void stage_rows_w(float* dst, const float* src_base, long row0_off, long tok_stride, int first, int n, int L) {
    for (int idx = threadIdx.x; idx < n * 4; idx += NTH) {
        int r = idx >> 2, q4 = idx & 3;
        int tok = first + r;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (tok >= 0 && tok < L) v = __ldg(reinterpret_cast<const float4*>(src_base + (row0_off + (long)tok * tok_stride) * LDQ) + q4);
        *reinterpret_cast<float4*>(dst + r * WLD + q4 * 4) = v;
    }
}
// E window: row w holds E[clamp(rfirst + w) + 512]
__device__ __forceinline__ void stage_E(float* dst, const float* E, int rfirst, int n) {
    for (int idx = threadIdx.x; idx < n * 4; idx += NTH) {
        int w = idx >> 2, q4 = idx & 3;
        int e = clampi(rfirst + w, -MAXPOS, MAXPOS) + MAXPOS;
        *reinterpret_cast<float4*>(dst + w * WLD + q4 * 4) = __ldg(reinterpret_cast<const float4*>(E + e * D) + q4);
    }
}

// ------------------------------------------------------------------------------------------ forward
// VAR: ragged batch (frames, axis; common.cuh): a sequence's length is its own (time axis) and sequences of padded frames do no work
// (frequency axis), so a valid row is computed with exactly the arithmetic of a run on its utterance alone.
template <bool VAR>
__global__ void __launch_bounds__(NTH) attn_fwd_kernel(const float* __restrict__ qkv, SeqGeom g, const float* __restrict__ E,
                                                       float* __restrict__ ctx, float* __restrict__ lse, const int* __restrict__ frames,
                                                       int axis) {
    __shared__ __align__(16) float Ks[TILE * D], Vs[TILE * D], Es[WROWS * WLD];
    const int s = blockIdx.x / H, h = blockIdx.x % H;
    const int i0 = blockIdx.y * NTH, il = threadIdx.x, i = i0 + il;
    const int L = VAR ? varlen_seq_len(g, frames, axis, s) : g.L;
    if (VAR && i0 >= L) return;
    const long base = seq_base(g, s);
    const bool active = i < L;
    float q[D], acc[D];
#pragma unroll
    for (int d = 0; d < D; ++d) { q[d] = 0.f; acc[d] = 0.f; }
    if (active) {
        ld16(qkv + (base + (long)i * g.tok_stride) * LDQ + h * D, q);
#pragma unroll
        for (int d = 0; d < D; ++d) q[d] *= SCALE_LOG2E;
    }
    float mrun = -INFINITY, lrun = 0.f;
    for (int j0 = 0; j0 < L; j0 += TILE) {
        const int nk = min(TILE, L - j0);
        __syncthreads();
        stage_rows16(Ks, qkv + CQ + h * D, base, g.tok_stride, j0, nk, L, 1.f);
        stage_rows16(Vs, qkv + 2 * CQ + h * D, base, g.tok_stride, j0, nk, L, 1.f);
        // r = i - j = (i0 - j0) + (il - jl);  window row w = il - jl + TILE - 1
        stage_E(Es, E, i0 - j0 - (TILE - 1), NTH + nk - 1 + (TILE - nk));
        __syncthreads();
        for (int jc = 0; jc < nk; jc += 8) {
            float sc[8];
            float cmax = -INFINITY;
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                int jl = jc + u;
                float a = -INFINITY;
                if (jl < nk) {
                    const float* kp = Ks + jl * D;
                    const float* ep = Es + (il - jl + TILE - 1) * WLD;
                    a = 0.f;
#pragma unroll
                    for (int q4 = 0; q4 < 4; ++q4) {
                        float4 kk = *reinterpret_cast<const float4*>(kp + 4 * q4);
                        float4 ee = *reinterpret_cast<const float4*>(ep + 4 * q4);
                        a = fmaf(q[4 * q4], kk.x + ee.x, a); a = fmaf(q[4 * q4 + 1], kk.y + ee.y, a);
                        a = fmaf(q[4 * q4 + 2], kk.z + ee.z, a); a = fmaf(q[4 * q4 + 3], kk.w + ee.w, a);
                    }
                }
                sc[u] = a; cmax = fmaxf(cmax, a);
            }
            float mnew = fmaxf(mrun, cmax);
            float corr = exp2f(mrun - mnew);          // mrun = -inf on the first chunk -> 0
            lrun *= corr;
#pragma unroll
            for (int d = 0; d < D; ++d) acc[d] *= corr;
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                int jl = jc + u;
                if (jl < nk) {
                    float p = exp2f(sc[u] - mnew);
                    lrun += p;
                    const float* vp = Vs + jl * D;
#pragma unroll
                    for (int q4 = 0; q4 < 4; ++q4) {
                        float4 vv = *reinterpret_cast<const float4*>(vp + 4 * q4);
                        acc[4 * q4] = fmaf(p, vv.x, acc[4 * q4]); acc[4 * q4 + 1] = fmaf(p, vv.y, acc[4 * q4 + 1]);
                        acc[4 * q4 + 2] = fmaf(p, vv.z, acc[4 * q4 + 2]); acc[4 * q4 + 3] = fmaf(p, vv.w, acc[4 * q4 + 3]);
                    }
                }
            }
            mrun = mnew;
        }
    }
    if (active) {
        float inv = 1.f / lrun;
#pragma unroll
        for (int d = 0; d < D; ++d) acc[d] *= inv;
        long row = base + (long)i * g.tok_stride;
        st16(ctx + row * CQ + h * D, acc);
        if (lse) lse[row * H + h] = mrun + log2f(lrun);
    }
}

// ------------------------------------------------------------------------------------------ backward: dq (+ delta)
// delta[row, h] = sum_d dctx * ctx;  dq_i = 0.25 * sum_j ds_ij (k_j + e_ij),  ds = p (dp - delta), dp = dctx_i . v_j
__global__ void __launch_bounds__(NTH) attn_bwd_dq_kernel(const float* __restrict__ qkv, SeqGeom g, const float* __restrict__ E,
                                                          const float* __restrict__ ctx, const float* __restrict__ dctx,
                                                          const float* __restrict__ lse, float* __restrict__ delta,
                                                          float* __restrict__ dqkv) {
    __shared__ __align__(16) float Ks[TILE * D], Vs[TILE * D], Es[WROWS * WLD];
    const int s = blockIdx.x / H, h = blockIdx.x % H;
    const int i0 = blockIdx.y * NTH, il = threadIdx.x, i = i0 + il;
    const long base = seq_base(g, s);
    const bool active = i < g.L;
    const long row = base + (long)(active ? i : 0) * g.tok_stride;
    float q[D], dO[D], dq[D];
    float dl = 0.f, ls = 0.f;
#pragma unroll
    for (int d = 0; d < D; ++d) { q[d] = 0.f; dO[d] = 0.f; dq[d] = 0.f; }
    if (active) {
        float o[D];
        ld16(qkv + row * LDQ + h * D, q);
        ld16(dctx + row * CQ + h * D, dO);
        ld16(ctx + row * CQ + h * D, o);
#pragma unroll
        for (int d = 0; d < D; ++d) { q[d] *= SCALE_LOG2E; dl = fmaf(dO[d], o[d], dl); }
        ls = lse[row * H + h];
        delta[row * H + h] = dl;
    }
    for (int j0 = 0; j0 < g.L; j0 += TILE) {
        const int nk = min(TILE, g.L - j0);
        __syncthreads();
        stage_rows16(Ks, qkv + CQ + h * D, base, g.tok_stride, j0, nk, g.L, 1.f);
        stage_rows16(Vs, qkv + 2 * CQ + h * D, base, g.tok_stride, j0, nk, g.L, 1.f);
        stage_E(Es, E, i0 - j0 - (TILE - 1), WROWS);
        __syncthreads();
        if (!active) continue;
        for (int jl = 0; jl < nk; ++jl) {
            const float* kp = Ks + jl * D;
            const float* vp = Vs + jl * D;
            const float* ep = Es + (il - jl + TILE - 1) * WLD;
            float ke[D];
            float a = 0.f, dp = 0.f;
#pragma unroll
            for (int q4 = 0; q4 < 4; ++q4) {
                float4 kk = *reinterpret_cast<const float4*>(kp + 4 * q4);
                float4 ee = *reinterpret_cast<const float4*>(ep + 4 * q4);
                float4 vv = *reinterpret_cast<const float4*>(vp + 4 * q4);
                ke[4 * q4] = kk.x + ee.x; ke[4 * q4 + 1] = kk.y + ee.y; ke[4 * q4 + 2] = kk.z + ee.z; ke[4 * q4 + 3] = kk.w + ee.w;
                dp = fmaf(dO[4 * q4], vv.x, dp); dp = fmaf(dO[4 * q4 + 1], vv.y, dp);
                dp = fmaf(dO[4 * q4 + 2], vv.z, dp); dp = fmaf(dO[4 * q4 + 3], vv.w, dp);
            }
#pragma unroll
            for (int d = 0; d < D; ++d) a = fmaf(q[d], ke[d], a);
            float ds = exp2f(a - ls) * (dp - dl);
#pragma unroll
            for (int d = 0; d < D; ++d) dq[d] = fmaf(ds, ke[d], dq[d]);
        }
    }
    if (active) {
#pragma unroll
        for (int d = 0; d < D; ++d) dq[d] *= 0.25f;
        st16(dqkv + row * LDQ + h * D, dq);
    }
}

// ------------------------------------------------------------------------------------------ backward: dk, dv
// thread = key j.  dv_j = sum_i p_ij dctx_i;  dk_j = 0.25 * sum_i ds_ij q_i
__global__ void __launch_bounds__(NTH) attn_bwd_dkv_kernel(const float* __restrict__ qkv, SeqGeom g, const float* __restrict__ E,
                                                           const float* __restrict__ dctx, const float* __restrict__ lse,
                                                           const float* __restrict__ delta, float* __restrict__ dqkv) {
    __shared__ __align__(16) float Qs[TILE * D], Os[TILE * D], Es[WROWS * WLD];
    __shared__ float Ls[TILE], Dl[TILE];
    const int s = blockIdx.x / H, h = blockIdx.x % H;
    const int j0 = blockIdx.y * NTH, jl = threadIdx.x, j = j0 + jl;
    const long base = seq_base(g, s);
    const bool active = j < g.L;
    const long row = base + (long)(active ? j : 0) * g.tok_stride;
    float k[D], v[D], dk[D], dv[D];
#pragma unroll
    for (int d = 0; d < D; ++d) { k[d] = 0.f; v[d] = 0.f; dk[d] = 0.f; dv[d] = 0.f; }
    if (active) { ld16(qkv + row * LDQ + CQ + h * D, k); ld16(qkv + row * LDQ + 2 * CQ + h * D, v); }
    for (int i0 = 0; i0 < g.L; i0 += TILE) {
        const int nq = min(TILE, g.L - i0);
        __syncthreads();
        stage_rows16(Qs, qkv + h * D, base, g.tok_stride, i0, nq, g.L, SCALE_LOG2E);
        // dctx has 64-float rows: stage manually
        for (int idx = threadIdx.x; idx < nq * 4; idx += NTH) {
            int r = idx >> 2, q4 = idx & 3;
            long rr = base + (long)(i0 + r) * g.tok_stride;
            *reinterpret_cast<float4*>(Os + r * D + q4 * 4) = __ldg(reinterpret_cast<const float4*>(dctx + rr * CQ + h * D) + q4);
        }
        for (int r = threadIdx.x; r < nq; r += NTH) {
            long rr = base + (long)(i0 + r) * g.tok_stride;
            Ls[r] = lse[rr * H + h]; Dl[r] = delta[rr * H + h];
        }
        // r = i - j = (i0 - j0) + (iq - jl);  window row w = iq - jl + NTH - 1
        stage_E(Es, E, i0 - j0 - (NTH - 1), WROWS);
        __syncthreads();
        if (!active) continue;
        for (int iq = 0; iq < nq; ++iq) {
            const float* qp = Qs + iq * D;
            const float* op = Os + iq * D;
            const float* ep = Es + (iq - jl + NTH - 1) * WLD;
            float a = 0.f, dp = 0.f;
            float qq[D], oo[D];
#pragma unroll
            for (int q4 = 0; q4 < 4; ++q4) {
                float4 qv = *reinterpret_cast<const float4*>(qp + 4 * q4);
                float4 ov = *reinterpret_cast<const float4*>(op + 4 * q4);
                float4 ee = *reinterpret_cast<const float4*>(ep + 4 * q4);
                qq[4 * q4] = qv.x; qq[4 * q4 + 1] = qv.y; qq[4 * q4 + 2] = qv.z; qq[4 * q4 + 3] = qv.w;
                oo[4 * q4] = ov.x; oo[4 * q4 + 1] = ov.y; oo[4 * q4 + 2] = ov.z; oo[4 * q4 + 3] = ov.w;
                a = fmaf(qv.x, k[4 * q4] + ee.x, a); a = fmaf(qv.y, k[4 * q4 + 1] + ee.y, a);
                a = fmaf(qv.z, k[4 * q4 + 2] + ee.z, a); a = fmaf(qv.w, k[4 * q4 + 3] + ee.w, a);
            }
#pragma unroll
            for (int d = 0; d < D; ++d) dp = fmaf(oo[d], v[d], dp);
            float p = exp2f(a - Ls[iq]);
            float ds = p * (dp - Dl[iq]);
#pragma unroll
            for (int d = 0; d < D; ++d) { dv[d] = fmaf(p, oo[d], dv[d]); dk[d] = fmaf(ds, qq[d], dk[d]); }
        }
    }
    if (active) {
#pragma unroll
        for (int d = 0; d < D; ++d) dk[d] *= LN2;     // q was pre-scaled by 0.25*log2(e)
        st16(dqkv + row * LDQ + CQ + h * D, dk);
        st16(dqkv + row * LDQ + 2 * CQ + h * D, dv);
    }
}

// ------------------------------------------------------------------------------------------ backward: dE
// thread = (unclamped) relative distance rr = i - j.  dE[clamp(rr)+512] += 0.25 * sum_{seq, head, i} ds_{i, i-rr} q_i
__global__ void __launch_bounds__(NTH) attn_bwd_dE_kernel(const float* __restrict__ qkv, SeqGeom g, const float* __restrict__ E,
                                                          const float* __restrict__ dctx, const float* __restrict__ lse,
                                                          const float* __restrict__ delta, int seqs_per_block,
                                                          float* __restrict__ dE) {
    __shared__ __align__(16) float Qs[TILE * D], Os[TILE * D], Kw[WROWS * WLD], Vw[WROWS * WLD];
    __shared__ float Ls[TILE], Dl[TILE];
    const int r0 = (int)blockIdx.y * NTH - (g.L - 1);
    const int rl = threadIdx.x, rr = r0 + rl;
    const bool active = rr <= g.L - 1;
    const int eidx = clampi(rr, -MAXPOS, MAXPOS) + MAXPOS;
    float e[D], acc[D];
    ld16(E + eidx * D, e);
#pragma unroll
    for (int d = 0; d < D; ++d) acc[d] = 0.f;
    const int s_beg = blockIdx.x * seqs_per_block;
    const int s_end = min(s_beg + seqs_per_block, g.n_seq);
    for (int sh = s_beg * H; sh < s_end * H; ++sh) {
        const int s = sh / H, h = sh % H;
        const long base = seq_base(g, s);
        for (int i0 = 0; i0 < g.L; i0 += TILE) {
            const int nq = min(TILE, g.L - i0);
            // block-uniform skip: is any (i, rr) of this tile a valid pair (0 <= i - rr < L)?
            if (i0 + nq - 1 - r0 < 0 || i0 - (r0 + NTH - 1) > g.L - 1) continue;
            __syncthreads();
            stage_rows16(Qs, qkv + h * D, base, g.tok_stride, i0, nq, g.L, SCALE_LOG2E);
            for (int idx = threadIdx.x; idx < nq * 4; idx += NTH) {
                int r = idx >> 2, q4 = idx & 3;
                long rw = base + (long)(i0 + r) * g.tok_stride;
                *reinterpret_cast<float4*>(Os + r * D + q4 * 4) = __ldg(reinterpret_cast<const float4*>(dctx + rw * CQ + h * D) + q4);
            }
            for (int r = threadIdx.x; r < nq; r += NTH) {
                long rw = base + (long)(i0 + r) * g.tok_stride;
                Ls[r] = lse[rw * H + h]; Dl[r] = delta[rw * H + h];
            }
            // j = i - rr = (i0 - r0) + (iq - rl);  window row w = iq - rl + NTH - 1  ->  j = jfirst + w
            const int jfirst = i0 - r0 - (NTH - 1);
            stage_rows_w(Kw, qkv + CQ + h * D, base, g.tok_stride, jfirst, WROWS, g.L);
            stage_rows_w(Vw, qkv + 2 * CQ + h * D, base, g.tok_stride, jfirst, WROWS, g.L);
            __syncthreads();
            if (!active) continue;
            for (int iq = 0; iq < nq; ++iq) {
                const int w = iq - rl + NTH - 1;
                const int j = jfirst + w;
                if (j < 0 || j >= g.L) continue;
                const float* qp = Qs + iq * D;
                const float* op = Os + iq * D;
                const float* kp = Kw + w * WLD;
                const float* vp = Vw + w * WLD;
                float a = 0.f, dp = 0.f;
                float qq[D];
#pragma unroll
                for (int q4 = 0; q4 < 4; ++q4) {
                    float4 qv = *reinterpret_cast<const float4*>(qp + 4 * q4);
                    float4 ov = *reinterpret_cast<const float4*>(op + 4 * q4);
                    float4 kk = *reinterpret_cast<const float4*>(kp + 4 * q4);
                    float4 vv = *reinterpret_cast<const float4*>(vp + 4 * q4);
                    qq[4 * q4] = qv.x; qq[4 * q4 + 1] = qv.y; qq[4 * q4 + 2] = qv.z; qq[4 * q4 + 3] = qv.w;
                    a = fmaf(qv.x, kk.x + e[4 * q4], a); a = fmaf(qv.y, kk.y + e[4 * q4 + 1], a);
                    a = fmaf(qv.z, kk.z + e[4 * q4 + 2], a); a = fmaf(qv.w, kk.w + e[4 * q4 + 3], a);
                    dp = fmaf(ov.x, vv.x, dp); dp = fmaf(ov.y, vv.y, dp); dp = fmaf(ov.z, vv.z, dp); dp = fmaf(ov.w, vv.w, dp);
                }
                float ds = exp2f(a - Ls[iq]) * (dp - Dl[iq]);
#pragma unroll
                for (int d = 0; d < D; ++d) acc[d] = fmaf(ds, qq[d], acc[d]);
            }
        }
    }
    if (active) {
#pragma unroll
        for (int d = 0; d < D; ++d) atomicAdd(dE + eidx * D + d, acc[d] * LN2);
    }
}

}  // namespace

static SeqGeom geom_from(int B, int T, int F, int axis) { return make_seq_geom(B, T, F, axis); }

// qkv (B*T*F, 192) -> ctx (B*T*F, 64), lse (B*T*F, 4) (base-2 log-sum-exp of the scaled logits; may be null).
// axis 0: sequences along T (time conformer, generator.py:94); axis 1: along F (freq conformer, generator.py:96).
// frames (optional, device int[B]): ragged batch; rows of padded frames are neither read nor written.
static int attention_fwd_launch(const float* qkv, const float* E, int B, int T, int F, int axis, const int* frames, float* ctx, float* lse,
                                void* stream) {
    CMGAN_REQUIRE(qkv && E && ctx, "cmgan_attention_fwd: null pointer");
    CMGAN_REQUIRE(axis == 0 || axis == 1, "cmgan_attention_fwd: axis must be 0 (time) or 1 (freq)");
    SeqGeom g = geom_from(B, T, F, axis);
    if (g.n_seq == 0 || g.L == 0) return 0;
    dim3 grid(g.n_seq * H, cdiv(g.L, NTH));
    if (frames) attn_fwd_kernel<true><<<grid, NTH, 0, (cudaStream_t)stream>>>(qkv, g, E, ctx, lse, frames, axis);
    else attn_fwd_kernel<false><<<grid, NTH, 0, (cudaStream_t)stream>>>(qkv, g, E, ctx, lse, nullptr, axis);
    return cmgan_check_launch("attn_fwd_kernel");
}

CMGAN_API int cmgan_attention_fwd(const float* qkv, const float* E, int B, int T, int F, int axis, float* ctx, float* lse, void* stream) {
    return attention_fwd_launch(qkv, E, B, T, F, axis, nullptr, ctx, lse, stream);
}

CMGAN_API int cmgan_attention_fwd_varlen(const float* qkv, const float* E, int B, int T, int F, int axis, const int* frames, float* ctx, float* lse,
                                         void* stream) {
    CMGAN_REQUIRE(frames, "cmgan_attention_fwd_varlen: null frames");
    return attention_fwd_launch(qkv, E, B, T, F, axis, frames, ctx, lse, stream);
}

// dqkv (B*T*F, 192) fully overwritten; dE (1025, 16) accumulated (+=); delta (B*T*F, 4) scratch.
CMGAN_API int cmgan_attention_bwd(const float* qkv, const float* E, const float* ctx, const float* dctx, const float* lse, int B, int T,
                                  int F, int axis, float* delta, float* dqkv, float* dE, void* stream) {
    CMGAN_REQUIRE(qkv && E && ctx && dctx && lse && delta && dqkv && dE, "cmgan_attention_bwd: null pointer");
    CMGAN_REQUIRE(axis == 0 || axis == 1, "cmgan_attention_bwd: axis must be 0 (time) or 1 (freq)");
    SeqGeom g = geom_from(B, T, F, axis);
    if (g.n_seq == 0 || g.L == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    dim3 grid(g.n_seq * H, cdiv(g.L, NTH));
    attn_bwd_dq_kernel<<<grid, NTH, 0, st>>>(qkv, g, E, ctx, dctx, lse, delta, dqkv);
    if (cmgan_check_launch("attn_bwd_dq_kernel")) return -1;
    attn_bwd_dkv_kernel<<<grid, NTH, 0, st>>>(qkv, g, E, dctx, lse, delta, dqkv);
    if (cmgan_check_launch("attn_bwd_dkv_kernel")) return -1;
    const int spb = 1;      // one sequence (x 4 heads) per block: enough blocks to fill the GPU; 16 red.global per thread at the end
    dim3 gridE(cdiv(g.n_seq, spb), cdiv(2 * g.L - 1, NTH));
    attn_bwd_dE_kernel<<<gridE, NTH, 0, st>>>(qkv, g, E, dctx, lse, delta, spb, dE);
    return cmgan_check_launch("attn_bwd_dE_kernel");
}
