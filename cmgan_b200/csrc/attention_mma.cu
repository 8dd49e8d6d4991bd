// Tensor-core (tf32 mma.sync) forward of the relative-position attention, flash style.  Same contract as attn_fwd_kernel in
// attention.cu (which stays the exact-fp32 path): qkv (M, 192) -> ctx (M, 64), lse (M, 4).
//
// One warp owns 16 queries of one (sequence, head); a block = 4 warps = 64 queries; keys are visited in tiles of 64.
// Per key tile and warp:   S  = Q K^T                       16 x 64   (16 mma.m16n8k8, K = head dim 16)
//                          R  = Q E_win^T                   16 x 80   relative-position logits for every distance the tile
//                                                                    can see; written to shared memory and read back skewed:
//                          S[i, j] += R[i, i - j]
//                          online softmax in the accumulator layout (row max / sum across the 4 lanes of a quad)
//                          O += P V                         P re-used in place as the A operand: the accumulator layout
//                                                           (cols 2t, 2t+1) equals the A layout (k = t, t+4) under a fixed
//                                                           permutation of the 8 keys of a k-step, applied to V's rows instead.
// Operands are rounded to tf32 when staged; accumulation, softmax and the running statistics are fp32.
#include <type_traits>

#include "common.cuh"
#include "../../include/cmgan_b200.h"
#include "tc_ptx.cuh"

namespace {
using cmgan_tc::cp_async16;
using cmgan_tc::cp_async_commit;
using cmgan_tc::cp_async_wait;
using cmgan_tc::smem_u32;

constexpr int D = 16, H = 4, CQ = 64, LDQ = 192;
constexpr int QB = 64;            // queries per block (4 warps x 16)
constexpr int KT = 64;            // keys per tile
constexpr int LDS_ = 20;          // smem row stride of the 16-float operand rows (conflict-free fragment loads)
constexpr int EW = QB + KT - 1;   // 127 relative distances visible to a block per key tile
constexpr int RW = 80;            // relative distances visible to one warp (16 + 64 - 1 = 79, padded to 10 n-tiles)
constexpr int LDR = 84;
constexpr int MAXPOS = 512;
constexpr float SCALE_LOG2E = 0.25f * 1.4426950408889634f;

__device__ __forceinline__ float tf32r(float x) {
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
    return __uint_as_float(r);
}
// tf32 rounding of a finite value in one integer add: the tensor core ignores the low 13 mantissa bits, so adding half a tf32 ulp to the
// bit pattern first makes that truncation a round-to-nearest (ties away from zero) -- cvt.rna.tf32.f32 costs five instructions here
__device__ __forceinline__ float tf32q(float x) { return __uint_as_float(__float_as_uint(x) + 0x1000u); }
// 2^x on the raw MUFU approximation (exp2f wraps it in range handling a softmax argument <= 0 does not need)
__device__ __forceinline__ float ex2(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ void mma_tf32(float c[4], const float a[4], float b0, float b1) {
    asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
                 : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
                 : "r"(__float_as_uint(a[0])), "r"(__float_as_uint(a[1])), "r"(__float_as_uint(a[2])), "r"(__float_as_uint(a[3])),
                   "r"(__float_as_uint(b0)), "r"(__float_as_uint(b1)));
}
__device__ __forceinline__ int clampi(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }

// One tile of operands, staged asynchronously (cp.async, 16 B, zero fill past the end of the sequence) one tile ahead of its use:
//   As, Bs : 64 rows x 16 floats (row stride LDS_) of two row operands (K and V, or Q and dO), rows first .. first + 63 of the sequence
//   Es     : the relative-position rows E[clamp(rfirst + w)] for w < EROWS
// Raw fp32 lands in shared memory; the tensor cores read the tf32 bits of it (low mantissa bits ignored).
constexpr int EROWS = EW + 1;     // 128: every window row an n-tile can touch
constexpr int TILE_FLOATS = 2 * KT * LDS_ + EROWS * LDS_;
__device__ __forceinline__ void stage_tile_async(float* buf, const float* __restrict__ a_src, int a_ld, const float* __restrict__ b_src, int b_ld,
                                                 long base, long tok_stride, int first, int L, const float* __restrict__ E, int rfirst, int tid) {
    const uint32_t sa = smem_u32(buf), sb = sa + KT * LDS_ * 4, se = sb + KT * LDS_ * 4;
    for (int idx = tid; idx < KT * 4; idx += 128) {
        const int r = idx >> 2, q4 = idx & 3;
        const bool ok = first + r < L;
        const long row = base + (long)(ok ? first + r : 0) * tok_stride;
        cp_async16(sa + (r * LDS_ + q4 * 4) * 4, a_src + row * a_ld + q4 * 4, ok ? 16u : 0u);
        cp_async16(sb + (r * LDS_ + q4 * 4) * 4, b_src + row * b_ld + q4 * 4, ok ? 16u : 0u);
    }
    for (int idx = tid; idx < EROWS * 4; idx += 128) {
        const int w = idx >> 2, q4 = idx & 3;
        const int e = clampi(rfirst + w, -MAXPOS, MAXPOS) + MAXPOS;
        cp_async16(se + (w * LDS_ + q4 * 4) * 4, E + e * D + q4 * 4, 16u);
    }
}

// NBUF = 2: the next key tile is staged while the current one is processed (62.5 KB of shared memory, 3 blocks / SM).
// NBUF = 1: one tile buffer, staged and waited for at the top of each iteration (42 KB, 5 blocks / SM): the load latency is hidden by the
// other resident blocks instead of by a second buffer.
// VAR: ragged batch (frames, axis; common.cuh): the key and query length of a sequence is its own (time axis), sequences of padded
// frames do no work (frequency axis); a valid row gets exactly the arithmetic of a run on its utterance alone.
template <int NBUF, bool VAR>
__global__ void __launch_bounds__(128) attn_fwd_mma_kernel(const float* __restrict__ qkv, SeqGeom g, const float* __restrict__ E,
                                                           float* __restrict__ ctx, float* __restrict__ lse, const int* __restrict__ frames,
                                                           int axis) {
    extern __shared__ __align__(16) float smem_fwd[];          // tile buffers [NBUF][TILE_FLOATS] | Rs[4][16 * LDR]
    float* Rs0 = smem_fwd + NBUF * TILE_FLOATS;
    const int s = blockIdx.x / H, h = blockIdx.x % H;
    const int i0 = blockIdx.y * QB;
    const int L = VAR ? varlen_seq_len(g, frames, axis, s) : g.L;
    if (VAR && i0 >= L) return;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, gq = lane >> 2, t = lane & 3;
    const long base = seq_base(g, s);
    const int iw = i0 + warp * 16;                    // first query of this warp
    const bool warp_active = iw < L;

    // ---- Q fragments (rows gq, gq+8), scaled and rounded once
    float qa[2][4];
#pragma unroll
    for (int ks = 0; ks < 2; ++ks)
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const int row = iw + gq + (r & 1) * 8, col = t + (r >> 1) * 4 + ks * 8;
            float v = 0.f;
            if (row < L) v = __ldg(qkv + (base + (long)row * g.tok_stride) * LDQ + h * D + col) * SCALE_LOG2E;
            qa[ks][r] = tf32r(v);
        }
    float o[2][4];
#pragma unroll
    for (int nd = 0; nd < 2; ++nd)
#pragma unroll
        for (int r = 0; r < 4; ++r) o[nd][r] = 0.f;
    float mrun[2] = {-INFINITY, -INFINITY}, lrun[2] = {0.f, 0.f};     // rows gq and gq+8 (lrun: this lane's partial sum)

    const float* ksrc = qkv + h * D + CQ;
    const float* vsrc = qkv + h * D + 2 * CQ;
    // window row w <-> relative distance r = (i0 - j0 - (KT - 1)) + w
    if (NBUF == 2) {
        stage_tile_async(smem_fwd, ksrc, LDQ, vsrc, LDQ, base, g.tok_stride, 0, L, E, i0 - (KT - 1), tid);
        cp_async_commit();
    }
    for (int j0 = 0, it = 0; j0 < L; j0 += KT, ++it) {
        const int nk = min(KT, L - j0);
        const float* Ks = smem_fwd + (NBUF == 2 ? (it & 1) : 0) * TILE_FLOATS;
        const float* Vs = Ks + KT * LDS_;
        const float* Es = Vs + KT * LDS_;
        __syncthreads();                              // every warp is done with the buffer the next tile is staged into
        if (NBUF == 2) {
            if (j0 + KT < L)
                stage_tile_async(smem_fwd + ((it + 1) & 1) * TILE_FLOATS, ksrc, LDQ, vsrc, LDQ, base, g.tok_stride, j0 + KT, L, E,
                                 i0 - (j0 + KT) - (KT - 1), tid);
            cp_async_commit();
            cp_async_wait<1>();                       // this tile has landed (the group just committed may still be in flight)
        } else {
            stage_tile_async(smem_fwd, ksrc, LDQ, vsrc, LDQ, base, g.tok_stride, j0, L, E, i0 - j0 - (KT - 1), tid);
            cp_async_commit();
            cp_async_wait<0>();
        }
        __syncthreads();
        if (!warp_active) continue;
        // a full tile (64 valid keys) runs the straight-line path; the short last tile skips the n-tiles past its end
        auto tile_body = [&](auto full_tag) {
        constexpr bool FULL = decltype(full_tag)::value;
        const int ntv = (nk + 7) >> 3;          // key n-tiles that hold at least one valid key (a short last tile skips the rest)
        const int rt0 = (KT - nk) >> 3;         // first n-tile of relative distances a valid key can reach

        // ---- S = Q K^T
        float sc[8][4];
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
            sc[nt][0] = sc[nt][1] = sc[nt][2] = sc[nt][3] = 0.f;
            if (!FULL && nt >= ntv) continue;
#pragma unroll
            for (int ks = 0; ks < 2; ++ks) {
                const float* kp = Ks + (nt * 8 + gq) * LDS_ + t + ks * 8;
                mma_tf32(sc[nt], qa[ks], kp[0], kp[4]);
            }
        }
        // ---- R = Q E^T over this warp's 80 distances: window rows [16 w, 16 w + 80)   (r = iw - j0 - 63 + c)
        float* R = Rs0 + warp * 16 * LDR;
#pragma unroll
        for (int nt = 0; nt < RW / 8; ++nt) {
            if (!FULL && nt < rt0) continue;
            float rc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
            for (int ks = 0; ks < 2; ++ks) {
                const float* ep = Es + (warp * 16 + nt * 8 + gq) * LDS_ + t + ks * 8;
                mma_tf32(rc, qa[ks], ep[0], ep[4]);
            }
            *reinterpret_cast<float2*>(R + gq * LDR + nt * 8 + 2 * t) = make_float2(rc[0], rc[1]);
            *reinterpret_cast<float2*>(R + (gq + 8) * LDR + nt * 8 + 2 * t) = make_float2(rc[2], rc[3]);
        }
        __syncwarp();
        // ---- S[i, j] += R[i, i - j]:  column of (query row q, key column c) is q - c + 63
        float tmax[2] = {-INFINITY, -INFINITY};
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
            if (!FULL && nt >= ntv) { sc[nt][0] = sc[nt][1] = sc[nt][2] = sc[nt][3] = -INFINITY; continue; }
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                const int qrow = gq + (r >> 1) * 8, kcol = nt * 8 + 2 * t + (r & 1);
                float v = sc[nt][r] + R[qrow * LDR + qrow - kcol + (KT - 1)];
                if (!FULL && kcol >= nk) v = -INFINITY;
                sc[nt][r] = v;
                tmax[r >> 1] = fmaxf(tmax[r >> 1], v);
            }
        }
        __syncwarp();                 // R is rewritten in the next key tile
        // ---- online softmax (rows gq, gq+8): reduce over the quad
        float corr[2];
#pragma unroll
        for (int hrow = 0; hrow < 2; ++hrow) {
            float m = tmax[hrow];
            m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, 1));
            m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, 2));
            const float mnew = fmaxf(mrun[hrow], m);
            corr[hrow] = ex2(mrun[hrow] - mnew);
            mrun[hrow] = mnew;
            lrun[hrow] *= corr[hrow];
        }
#pragma unroll
        for (int nd = 0; nd < 2; ++nd) { o[nd][0] *= corr[0]; o[nd][1] *= corr[0]; o[nd][2] *= corr[1]; o[nd][3] *= corr[1]; }
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
            if (!FULL && nt >= ntv) continue;
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                const float p = ex2(sc[nt][r] - mrun[r >> 1]);
                lrun[r >> 1] += p;
                sc[nt][r] = tf32q(p);
            }
        }
        // ---- O += P V.  k-step kk covers keys 8 kk .. 8 kk + 7; A-operand column t <-> key 2t, column t+4 <-> key 2t+1
#pragma unroll
        for (int kk = 0; kk < 8; ++kk) {
            if (!FULL && kk >= ntv) continue;
            const float pa[4] = {sc[kk][0], sc[kk][2], sc[kk][1], sc[kk][3]};
#pragma unroll
            for (int nd = 0; nd < 2; ++nd) {
                const float* vp = Vs + (kk * 8 + 2 * t) * LDS_ + nd * 8 + gq;
                mma_tf32(o[nd], pa, vp[0], vp[LDS_]);
            }
        }
        };
        if (nk == KT) tile_body(std::true_type{}); else tile_body(std::false_type{});
    }
    if (!warp_active) return;
    // ---- finish: row sums across the quad, normalise, store
#pragma unroll
    for (int hrow = 0; hrow < 2; ++hrow) {
        float l = lrun[hrow];
        l += __shfl_xor_sync(0xffffffffu, l, 1);
        l += __shfl_xor_sync(0xffffffffu, l, 2);
        lrun[hrow] = l;
    }
#pragma unroll
    for (int hrow = 0; hrow < 2; ++hrow) {
        const int i = iw + gq + hrow * 8;
        if (i >= L) continue;
        const float inv = 1.f / lrun[hrow];
        const long row = base + (long)i * g.tok_stride;
#pragma unroll
        for (int nd = 0; nd < 2; ++nd)
            *reinterpret_cast<float2*>(ctx + row * CQ + h * D + nd * 8 + 2 * t) = make_float2(tf32r(o[nd][hrow * 2] * inv), tf32r(o[nd][hrow * 2 + 1] * inv));
        if (lse && t == 0) lse[row * H + h] = mrun[hrow] + log2f(lrun[hrow]);
    }
}


// ============================================================================================ backward
// Both backward kernels recompute the logits tile by tile exactly as the forward does (tf32 operands, fp32 accumulate) and use
//   p = exp2(s - lse),  dp = dO V^T,  ds = p (dp - delta),  delta_i = dO_i . O_i
// (ds is the gradient wrt the natural-log logits; q is held pre-scaled by 0.25 log2(e), so sums against q take a final ln 2).
constexpr float LN2 = 0.6931471805599453f;

// ---- delta[row, h] = dO[row, h, :] . O[row, h, :]  (one thread per (row, head); lets the dq and dk/dv kernels run side by side)
__global__ void attn_delta_kernel(const float* __restrict__ ctx, const float* __restrict__ dctx, long n, float* __restrict__ delta) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float4* o = reinterpret_cast<const float4*>(ctx + i * D);
    const float4* d = reinterpret_cast<const float4*>(dctx + i * D);
    float acc = 0.f;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const float4 a = __ldg(o + k), b = __ldg(d + k);
        acc = fmaf(a.x, b.x, acc); acc = fmaf(a.y, b.y, acc); acc = fmaf(a.z, b.z, acc); acc = fmaf(a.w, b.w, acc);
    }
    delta[i] = acc;
}

// ---- dq, delta and dE.  A block owns one 64-query tile position and walks over many (sequence, head) items, so the relative
// distances it touches are the same for every item and dE can be accumulated in shared memory, flushed once at the end.
//   dQ  = dS K  +  dR E_win                 dR[i, c] = dS[i, j],  c = i_l - j_l + 63  (dS scattered skewed into the block's R buffer,
//                                           64 queries x 127 distances; a warp writes only its own 16 rows)
//   dEw = dR^T Q                            128 x 16 per block and key tile; each warp owns 32 distances -> plain adds into the
//                                           block accumulator (no atomics: shared fp32 atomics are CAS loops)
// dynamic smem: (Ks | Vs | Es)[2] | Rb[64 x LDRB] | Qs[64 x 20] | dEs[(Lpad + 64) x 16]
constexpr int LDRB = 136;
// GDE = false: the dE accumulator lives in shared memory next to two tile buffers (110 KB at L = 321: 2 blocks / SM, 1 at L = 1281).
// GDE = true : the accumulator is a block-private slab of global memory (L2-resident read-modify-write, no atomics: a block owns its slab) and
//              the K / V / E tile is single-buffered: 60 KB -> 3 blocks / SM at every L; the other resident blocks hide the tile loads.
template <bool GDE>
__global__ void __launch_bounds__(128, GDE ? 3 : 2) attn_bwd_dq_mma_kernel(const float* __restrict__ qkv, SeqGeom g, const float* __restrict__ E,
                                                              const float* __restrict__ ctx, const float* __restrict__ dctx,
                                                              const float* __restrict__ lse, int n_items, int Lpad,
                                                              float* __restrict__ delta, float* __restrict__ dqkv,
                                                              float* __restrict__ dE, float* __restrict__ de_scratch) {
    extern __shared__ __align__(16) float smem_dq[];
    constexpr int NBUF = GDE ? 1 : 2;
    float* Rb = smem_dq + NBUF * TILE_FLOATS;         // after the K / V / E tile buffer(s)
    float* Qs = Rb + QB * LDRB;
    float* dEs = GDE ? de_scratch + ((long)blockIdx.y * gridDim.x + blockIdx.x) * (long)(Lpad + 64) * D : Qs + QB * LDS_;
    const int i0 = blockIdx.y * QB;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, gq = lane >> 2, t = lane & 3;
    const int iw = i0 + warp * 16;
    const bool warp_active = iw < g.L;
    const int acc_rows = Lpad + 64;
    const int r_acc0 = i0 - Lpad + 1;                 // relative distance of accumulator row 0
    for (int idx = tid; idx < acc_rows * D; idx += 128) dEs[idx] = 0.f;
    for (int idx = tid; idx < QB * LDRB; idx += 128) Rb[idx] = 0.f;
    float* R = Rb + warp * 16 * LDRB + warp * 16;     // this warp's rows; its 80-distance window starts at block column 16 warp
    float* Qw = Qs + warp * 16 * LDS_;

    // tiles are staged one ahead, across item boundaries: (item, j0) -> (item, j0 + 64) or (next item, 0)
    auto stage = [&](int item, int j0, int slot) {
        const int s = item / H, h = item % H;
        stage_tile_async(smem_dq + slot * TILE_FLOATS, qkv + h * D + CQ, LDQ, qkv + h * D + 2 * CQ, LDQ, seq_base(g, s), g.tok_stride, j0, g.L, E,
                         i0 - j0 - (KT - 1), tid);
    };
    if (!GDE) {
        if ((int)blockIdx.x < n_items) stage(blockIdx.x, 0, 0);
        cp_async_commit();
    }
    int it = 0;
    // ---- per-item row operands: q (scaled), dO as A fragments; delta, lse for rows gq, gq + 8.  They are fetched one item ahead -- the
    // loads are issued while the previous item's last key tile is being processed -- so an item does not start by waiting for global memory
    // (that wait was 22 % of the kernel's stall samples: a sequence has only 2 - 6 key tiles to amortise it over).
    float qn[2][4], dn[2][4], dln[2], lsn[2];
    auto fetch_item = [&](int item) {
        const int s = item / H, h = item % H;
        const long base = seq_base(g, s);
#pragma unroll
        for (int ks = 0; ks < 2; ++ks)
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                const int row = iw + gq + (r & 1) * 8, col = t + (r >> 1) * 4 + ks * 8;
                float qv = 0.f, dv = 0.f;
                if (row < g.L) {
                    const long rr = base + (long)row * g.tok_stride;
                    qv = __ldg(qkv + rr * LDQ + h * D + col);
                    dv = __ldg(dctx + rr * CQ + h * D + col);
                }
                qn[ks][r] = qv;
                dn[ks][r] = dv;
            }
#pragma unroll
        for (int hrow = 0; hrow < 2; ++hrow) {
            const int row = iw + gq + hrow * 8;
            lsn[hrow] = 0.f; dln[hrow] = 0.f;
            if (row < g.L) {
                const long rr = base + (long)row * g.tok_stride;
                lsn[hrow] = __ldg(lse + rr * H + h);
                dln[hrow] = __ldg(delta + rr * H + h);          // written by attn_delta_kernel (the dk / dv kernel reads the same values)
            }
        }
    };
    if (!GDE && (int)blockIdx.x < n_items) fetch_item(blockIdx.x);
    for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
        const int s = item / H, h = item % H;
        const long base = seq_base(g, s);
        if (GDE) fetch_item(item);         // three resident blocks hide this latency; the prefetch registers would cost the third block
        float qa[2][4], da[2][4], dl[2], ls[2];
#pragma unroll
        for (int ks = 0; ks < 2; ++ks)
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                qa[ks][r] = tf32r(qn[ks][r] * SCALE_LOG2E);
                da[ks][r] = tf32r(dn[ks][r]);
            }
        dl[0] = dln[0]; dl[1] = dln[1]; ls[0] = lsn[0]; ls[1] = lsn[1];
        float dq[2][4];
#pragma unroll
        for (int nd = 0; nd < 2; ++nd)
#pragma unroll
            for (int r = 0; r < 4; ++r) dq[nd][r] = 0.f;

        for (int j0 = 0; j0 < g.L; j0 += KT) {
            const int nk = min(KT, g.L - j0);
            __syncthreads();               // previous tile's dE pass (reads Rb, Qs of every warp) is complete
            if (j0 == 0) {
#pragma unroll
                for (int ks = 0; ks < 2; ++ks)
#pragma unroll
                    for (int r = 0; r < 4; ++r) Qw[(gq + (r & 1) * 8) * LDS_ + t + (r >> 1) * 4 + ks * 8] = qa[ks][r];
            }
            if (GDE) {
                stage(item, j0, 0);
                cp_async_commit();
                cp_async_wait<0>();
            } else {
                if (j0 + KT < g.L) stage(item, j0 + KT, (it + 1) & 1);
                else if (item + (int)gridDim.x < n_items) {
                    stage(item + gridDim.x, 0, (it + 1) & 1);
                    fetch_item(item + gridDim.x);          // consumed when the next item starts
                }
                cp_async_commit();
                cp_async_wait<1>();
            }
            __syncthreads();
            const float* Ks = smem_dq + (GDE ? 0 : (it & 1)) * TILE_FLOATS;
            const float* Vs = Ks + KT * LDS_;
            const float* Es = Vs + KT * LDS_;
            ++it;
            auto tile_body = [&](auto full_tag) {       // full tile: straight-line; short last tile: skips the n-tiles past its end
            constexpr bool FULL = decltype(full_tag)::value;
            const int ntv = (nk + 7) >> 3;          // key n-tiles with at least one valid key
            const int rt0 = (KT - nk) >> 3;         // first 8-distance group a valid key can reach (window / block columns >= 64 - nk)
            if (warp_active) {
                // ---- S = Q K^T, dP = dO V^T
                float sc[8][4], dp[8][4];
#pragma unroll
                for (int nt = 0; nt < 8; ++nt) {
                    sc[nt][0] = sc[nt][1] = sc[nt][2] = sc[nt][3] = 0.f;
                    dp[nt][0] = dp[nt][1] = dp[nt][2] = dp[nt][3] = 0.f;
                    if (!FULL && nt >= ntv) continue;
#pragma unroll
                    for (int ks = 0; ks < 2; ++ks) {
                        const float* kp = Ks + (nt * 8 + gq) * LDS_ + t + ks * 8;
                        const float* vp = Vs + (nt * 8 + gq) * LDS_ + t + ks * 8;
                        mma_tf32(sc[nt], qa[ks], kp[0], kp[4]);
                        mma_tf32(dp[nt], da[ks], vp[0], vp[4]);
                    }
                }
                // ---- R = Q E_win^T -> smem (this warp's rows, window columns 0..79)
#pragma unroll
                for (int nt = 0; nt < RW / 8; ++nt) {
                    if (!FULL && nt < rt0) continue;
                    float rc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
                    for (int ks = 0; ks < 2; ++ks) {
                        const float* ep = Es + (warp * 16 + nt * 8 + gq) * LDS_ + t + ks * 8;
                        mma_tf32(rc, qa[ks], ep[0], ep[4]);
                    }
                    *reinterpret_cast<float2*>(R + gq * LDRB + nt * 8 + 2 * t) = make_float2(rc[0], rc[1]);
                    *reinterpret_cast<float2*>(R + (gq + 8) * LDRB + nt * 8 + 2 * t) = make_float2(rc[2], rc[3]);
                }
                __syncwarp();
                // ---- ds = exp2(s + R_skew - lse) (dp - delta), tf32
#pragma unroll
                for (int nt = 0; nt < 8; ++nt) {
                    if (!FULL && nt >= ntv) continue;            // sc stays 0: scattered below so that the band of dR is fully rewritten
#pragma unroll
                    for (int r = 0; r < 4; ++r) {
                        const int qrow = gq + (r >> 1) * 8, kcol = nt * 8 + 2 * t + (r & 1);
                        const float a = sc[nt][r] + R[qrow * LDRB + qrow - kcol + (KT - 1)];
                        float ds = ex2(a - ls[r >> 1]) * (dp[nt][r] - dl[r >> 1]);
                        if (!FULL && kcol >= nk) ds = 0.f;
                        sc[nt][r] = tf32q(ds);
                    }
                }
                __syncwarp();
                // ---- dR: scatter ds skewed into the same rows; the 16 window columns per row outside the band are zeroed
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    const int idx = lane + 32 * u, row = idx >> 4, c = (row + 64 + (idx & 15)) % RW;
                    R[row * LDRB + c] = 0.f;
                }
#pragma unroll
                for (int nt = 0; nt < 8; ++nt)
#pragma unroll
                    for (int r = 0; r < 4; ++r) {
                        const int qrow = gq + (r >> 1) * 8, kcol = nt * 8 + 2 * t + (r & 1);
                        R[qrow * LDRB + qrow - kcol + (KT - 1)] = sc[nt][r];
                    }
                __syncwarp();
                // ---- dQ += dS K   (A = dS re-used from the accumulator layout; keys of a k-step permuted, see forward)
#pragma unroll
                for (int kk = 0; kk < 8; ++kk) {
                    if (!FULL && kk >= ntv) continue;
                    const float pa[4] = {sc[kk][0], sc[kk][2], sc[kk][1], sc[kk][3]};
#pragma unroll
                    for (int nd = 0; nd < 2; ++nd) {
                        const float* kp = Ks + (kk * 8 + 2 * t) * LDS_ + nd * 8 + gq;
                        mma_tf32(dq[nd], pa, kp[0], kp[LDS_]);
                    }
                }
                // ---- dQ += dR E_win  (K = 80 distances)
#pragma unroll
                for (int kk = 0; kk < RW / 8; ++kk) {
                    if (!FULL && kk < rt0) continue;             // those distances only pair with keys past the end: dR = 0
                    const float ra[4] = {R[gq * LDRB + kk * 8 + t], R[(gq + 8) * LDRB + kk * 8 + t], R[gq * LDRB + kk * 8 + t + 4],
                                         R[(gq + 8) * LDRB + kk * 8 + t + 4]};
#pragma unroll
                    for (int nd = 0; nd < 2; ++nd) {
                        const float* ep = Es + (warp * 16 + kk * 8 + t) * LDS_ + nd * 8 + gq;
                        mma_tf32(dq[nd], ra, ep[0], ep[4 * LDS_]);
                    }
                }
            }
            __syncthreads();
            // ---- dE_win = dR^T Q over the block: M = 128 distances (32 per warp), K = 64 queries, N = 16
            {
                const int arow0 = (i0 - j0 - (KT - 1)) - r_acc0 + warp * 32;      // accumulator row of this warp's first distance
#pragma unroll
                for (int mt = 0; mt < 2; ++mt) {
                    if (!FULL && warp * 32 + mt * 16 + 16 <= KT - nk) continue;     // block columns below 64 - nk hold zeros only
                    float ec[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
#pragma unroll
                    for (int ks = 0; ks < QB / 8; ++ks) {
                        const float* rp = Rb + (t + 8 * ks) * LDRB + warp * 32 + 16 * mt + gq;
                        const float ta[4] = {rp[0], rp[8], rp[4 * LDRB], rp[4 * LDRB + 8]};
#pragma unroll
                        for (int nd = 0; nd < 2; ++nd) {
                            const float* qp = Qs + (t + 8 * ks) * LDS_ + nd * 8 + gq;
                            mma_tf32(ec[nd], ta, qp[0], qp[4 * LDS_]);
                        }
                    }
#pragma unroll
                    for (int nd = 0; nd < 2; ++nd)
#pragma unroll
                        for (int hrow = 0; hrow < 2; ++hrow) {
                            float2* ap = reinterpret_cast<float2*>(dEs + (arow0 + 16 * mt + gq + hrow * 8) * D + nd * 8 + 2 * t);
                            float2 v = *ap;
                            v.x += ec[nd][hrow * 2]; v.y += ec[nd][hrow * 2 + 1];
                            *ap = v;
                        }
                }
            }
            };
            if (nk == KT) tile_body(std::true_type{}); else tile_body(std::false_type{});
        }
        if (warp_active) {
#pragma unroll
            for (int hrow = 0; hrow < 2; ++hrow) {
                const int i = iw + gq + hrow * 8;
                if (i >= g.L) continue;
                const long row = base + (long)i * g.tok_stride;
#pragma unroll
                for (int nd = 0; nd < 2; ++nd)
                    *reinterpret_cast<float2*>(dqkv + row * LDQ + h * D + nd * 8 + 2 * t) =
                        make_float2(tf32r(0.25f * dq[nd][hrow * 2]), tf32r(0.25f * dq[nd][hrow * 2 + 1]));       // dqkv feeds two tensor-core contractions
            }
        }
    }
    __syncthreads();
    for (int idx = tid; idx < acc_rows * D; idx += 128) {
        const int rr = r_acc0 + idx / D;
        if (rr < -(g.L - 1) || rr > g.L - 1) continue;
        const float v = dEs[idx];
        if (v != 0.f) atomicAdd(dE + (clampi(rr, -MAXPOS, MAXPOS) + MAXPOS) * D + (idx % D), v * LN2);
    }
}

// ---- dk, dv.  One warp owns 16 keys; queries are visited in tiles of 64.  Everything is held transposed (rows = keys):
//   S^T = K Q^T + skew(R2),  R2 = Q_tile E_win^T (64 x 127, computed once per tile by the whole block)
//   dV += P^T dO,  dK += dS^T Q
constexpr int LDR2 = 132;
__global__ void __launch_bounds__(128, 3) attn_bwd_dkv_mma_kernel(const float* __restrict__ qkv, SeqGeom g, const float* __restrict__ E,
                                                               const float* __restrict__ dctx, const float* __restrict__ lse,
                                                               const float* __restrict__ delta, float* __restrict__ dqkv) {
    extern __shared__ __align__(16) float smem_kv[];
    float* R2 = smem_kv + 2 * TILE_FLOATS;            // after the two Q / dO / E tile buffers
    float* LD = R2 + QB * LDR2;                       // [2][lse (64) | delta (64)]
    const int s = blockIdx.x / H, h = blockIdx.x % H;
    const int j0 = blockIdx.y * KT;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, gq = lane >> 2, t = lane & 3;
    const long base = seq_base(g, s);
    const int jw = j0 + warp * 16;
    const bool warp_active = jw < g.L;

    float ka[2][4], va[2][4];
#pragma unroll
    for (int ks = 0; ks < 2; ++ks)
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const int row = jw + gq + (r & 1) * 8, col = t + (r >> 1) * 4 + ks * 8;
            float kv = 0.f, vv = 0.f;
            if (row < g.L) {
                const float* p = qkv + (base + (long)row * g.tok_stride) * LDQ + h * D + col;
                kv = __ldg(p + CQ);
                vv = __ldg(p + 2 * CQ);
            }
            ka[ks][r] = tf32r(kv * SCALE_LOG2E);       // the logit scale rides on K: Q is staged raw by cp.async
            va[ks][r] = tf32r(vv);
        }
    float dk[2][4], dv[2][4];
#pragma unroll
    for (int nd = 0; nd < 2; ++nd)
#pragma unroll
        for (int r = 0; r < 4; ++r) { dk[nd][r] = 0.f; dv[nd][r] = 0.f; }
    for (int idx = tid; idx < QB * LDR2; idx += 128) R2[idx] = 0.f;     // parts of R2 are skipped for short tiles but may be read (masked)

    const float* qsrc = qkv + h * D;
    const float* osrc = dctx + h * D;
    // lse / delta of the tile's queries: 4-byte cp.async (zero fill past the end; those queries are masked explicitly)
    auto stage = [&](int i0, int slot) {
        stage_tile_async(smem_kv + slot * TILE_FLOATS, qsrc, LDQ, osrc, CQ, base, g.tok_stride, i0, g.L, E, i0 - j0 - (KT - 1), tid);
        const int r = tid & 63;
        const bool ok = i0 + r < g.L;
        const long rr = base + (long)(ok ? i0 + r : 0) * g.tok_stride;
        const float* src = (tid < 64 ? lse : delta) + rr * H + h;
        asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(smem_u32(LD + slot * 2 * QB + tid)), "l"(src), "r"(ok ? 4u : 0u) : "memory");
    };
    stage(0, 0);
    cp_async_commit();
    for (int i0 = 0, it = 0; i0 < g.L; i0 += QB, ++it) {
        const int nq = min(QB, g.L - i0);
        __syncthreads();                                  // every warp is done with the buffers the next tile is staged into (and with R2)
        if (i0 + QB < g.L) stage(i0 + QB, (it + 1) & 1);
        cp_async_commit();
        cp_async_wait<1>();
        __syncthreads();
        const float* Qs = smem_kv + (it & 1) * TILE_FLOATS;       // window column c <-> distance (i0 - j0 - 63) + c,  c = il - jl + 63
        const float* Os = Qs + QB * LDS_;
        const float* Es = Os + QB * LDS_;
        const float* Ls = LD + (it & 1) * 2 * QB;
        const float* Dl = Ls + QB;
        auto tile_body = [&](auto full_tag) {           // full tile: straight-line; short last tile: skips the n-tiles past its end
        constexpr bool FULL = decltype(full_tag)::value;
        // ---- R2 rows 16 warp .. 16 warp + 15 (queries), all 128 window columns
        {
            float qa[2][4];
#pragma unroll
            for (int ks = 0; ks < 2; ++ks)
#pragma unroll
                for (int r = 0; r < 4; ++r) qa[ks][r] = Qs[(warp * 16 + gq + (r & 1) * 8) * LDS_ + t + (r >> 1) * 4 + ks * 8] * SCALE_LOG2E;
            // only rows of valid queries and the distances they can reach (columns <= nq + 62) are read back
            const int ntr = FULL ? 16 : (warp * 16 < nq ? min(16, ((nq + 62) >> 3) + 1) : 0);
#pragma unroll 4
            for (int nt = 0; nt < ntr; ++nt) {
                float rc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
                for (int ks = 0; ks < 2; ++ks) {
                    const float* ep = Es + (nt * 8 + gq) * LDS_ + t + ks * 8;
                    mma_tf32(rc, qa[ks], ep[0], ep[4]);
                }
                *reinterpret_cast<float2*>(R2 + (warp * 16 + gq) * LDR2 + nt * 8 + 2 * t) = make_float2(rc[0], rc[1]);
                *reinterpret_cast<float2*>(R2 + (warp * 16 + gq + 8) * LDR2 + nt * 8 + 2 * t) = make_float2(rc[2], rc[3]);
            }
        }
        __syncthreads();
        if (!warp_active) return;
        const int ntq = (nq + 7) >> 3;          // query n-tiles with at least one valid query

        // ---- S^T = K Q^T, dP^T = V dO^T     (rows = keys gq, gq+8 of this warp; columns = queries of the tile)
        float sc[8][4], dp[8][4];
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
            sc[nt][0] = sc[nt][1] = sc[nt][2] = sc[nt][3] = 0.f;
            dp[nt][0] = dp[nt][1] = dp[nt][2] = dp[nt][3] = 0.f;
            if (!FULL && nt >= ntq) continue;
#pragma unroll
            for (int ks = 0; ks < 2; ++ks) {
                const float* qp = Qs + (nt * 8 + gq) * LDS_ + t + ks * 8;
                const float* op = Os + (nt * 8 + gq) * LDS_ + t + ks * 8;
                mma_tf32(sc[nt], ka[ks], qp[0], qp[4]);
                mma_tf32(dp[nt], va[ks], op[0], op[4]);
            }
        }
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
            if (!FULL && nt >= ntq) continue;             // p = ds = 0 there (sc, dp still hold their zeros)
            const float2 l2 = *reinterpret_cast<const float2*>(Ls + nt * 8 + 2 * t);
            const float2 d2 = *reinterpret_cast<const float2*>(Dl + nt * 8 + 2 * t);
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                const int jl = warp * 16 + gq + (r >> 1) * 8, il = nt * 8 + 2 * t + (r & 1);
                const float a = sc[nt][r] + R2[il * LDR2 + il - jl + (KT - 1)];
                float p = ex2(a - ((r & 1) ? l2.y : l2.x));
                if (!FULL && il >= nq) p = 0.f;          // queries past the end of the sequence (their lse was zero-filled)
                sc[nt][r] = tf32q(p);
                dp[nt][r] = tf32q(p * (dp[nt][r] - ((r & 1) ? d2.y : d2.x)));
            }
        }
        // ---- dV += P^T dO,  dK += dS^T Q   (A from the accumulator layout; queries of a k-step permuted)
#pragma unroll
        for (int kk = 0; kk < 8; ++kk) {
            if (!FULL && kk >= ntq) continue;
            const float pa[4] = {sc[kk][0], sc[kk][2], sc[kk][1], sc[kk][3]};
            const float sa[4] = {dp[kk][0], dp[kk][2], dp[kk][1], dp[kk][3]};
#pragma unroll
            for (int nd = 0; nd < 2; ++nd) {
                const float* op = Os + (kk * 8 + 2 * t) * LDS_ + nd * 8 + gq;
                const float* qp = Qs + (kk * 8 + 2 * t) * LDS_ + nd * 8 + gq;
                mma_tf32(dv[nd], pa, op[0], op[LDS_]);
                mma_tf32(dk[nd], sa, qp[0], qp[LDS_]);
            }
        }
        };
        if (nq == QB) tile_body(std::true_type{}); else tile_body(std::false_type{});
    }
    if (!warp_active) return;
#pragma unroll
    for (int hrow = 0; hrow < 2; ++hrow) {
        const int j = jw + gq + hrow * 8;
        if (j >= g.L) continue;
        float* p = dqkv + (base + (long)j * g.tok_stride) * LDQ + h * D + 2 * t;
#pragma unroll
        for (int nd = 0; nd < 2; ++nd) {
            *reinterpret_cast<float2*>(p + CQ + nd * 8) = make_float2(tf32r(0.25f * dk[nd][hrow * 2]), tf32r(0.25f * dk[nd][hrow * 2 + 1]));      // Q was staged unscaled
            *reinterpret_cast<float2*>(p + 2 * CQ + nd * 8) = make_float2(tf32r(dv[nd][hrow * 2]), tf32r(dv[nd][hrow * 2 + 1]));
        }
    }
}

}  // namespace

// tf32 tensor-core forward (same outputs as cmgan_attention_fwd; logits carry tf32 operand rounding)
constexpr int FWD_NBUF_DEFAULT = 1;      // measured: 318 -> 280 us (time axis), 150 -> 138 us (frequency axis) at B = 4
CMGAN_API int cmgan_attention_fwd_tf32(const float* qkv, const float* E, int B, int T, int F, int axis, float* ctx, float* lse, void* stream) {
    return cmgan_attention_fwd_tf32_nbuf(qkv, E, B, T, F, axis, ctx, lse, FWD_NBUF_DEFAULT, stream);
}

// nbuf = 2: double-buffered key tiles, 3 blocks / SM; nbuf = 1: single buffer, 5 blocks / SM (see attn_fwd_mma_kernel)
CMGAN_API int cmgan_attention_fwd_tf32_nbuf(const float* qkv, const float* E, int B, int T, int F, int axis, float* ctx, float* lse, int nbuf,
                                            void* stream) {
    CMGAN_REQUIRE(qkv && E && ctx, "cmgan_attention_fwd_tf32: null pointer");
    CMGAN_REQUIRE(nbuf == 1 || nbuf == 2, "cmgan_attention_fwd_tf32_nbuf: nbuf must be 1 or 2");
    CMGAN_REQUIRE(axis == 0 || axis == 1, "cmgan_attention_fwd_tf32: axis must be 0 (time) or 1 (freq)");
    SeqGeom g = make_seq_geom(B, T, F, axis);
    if (g.n_seq == 0 || g.L == 0) return 0;
    dim3 grid(g.n_seq * H, cdiv(g.L, QB));
    const int smem = (nbuf * TILE_FLOATS + 4 * 16 * LDR) * (int)sizeof(float);
    static bool attr_set = false;
    if (!attr_set) {
        cudaError_t e = cudaFuncSetAttribute(attn_fwd_mma_kernel<2, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (2 * TILE_FLOATS + 4 * 16 * LDR) * (int)sizeof(float));
        CMGAN_REQUIRE(e == cudaSuccess, "cmgan_attention_fwd_tf32: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
        attr_set = true;
    }
    if (nbuf == 2) attn_fwd_mma_kernel<2, false><<<grid, 128, smem, (cudaStream_t)stream>>>(qkv, g, E, ctx, lse, nullptr, axis);
    else attn_fwd_mma_kernel<1, false><<<grid, 128, smem, (cudaStream_t)stream>>>(qkv, g, E, ctx, lse, nullptr, axis);
    return cmgan_check_launch("attn_fwd_mma_kernel");
}

// ragged batch (frames: device int[B], 1 <= frames[b] <= T): rows of padded frames are neither read nor written
CMGAN_API int cmgan_attention_fwd_tf32_varlen(const float* qkv, const float* E, int B, int T, int F, int axis, const int* frames, float* ctx,
                                              float* lse, void* stream) {
    CMGAN_REQUIRE(qkv && E && ctx && frames, "cmgan_attention_fwd_tf32_varlen: null pointer");
    CMGAN_REQUIRE(axis == 0 || axis == 1, "cmgan_attention_fwd_tf32_varlen: axis must be 0 (time) or 1 (freq)");
    SeqGeom g = make_seq_geom(B, T, F, axis);
    if (g.n_seq == 0 || g.L == 0) return 0;
    dim3 grid(g.n_seq * H, cdiv(g.L, QB));
    const int smem = (FWD_NBUF_DEFAULT * TILE_FLOATS + 4 * 16 * LDR) * (int)sizeof(float);
    attn_fwd_mma_kernel<FWD_NBUF_DEFAULT, true><<<grid, 128, smem, (cudaStream_t)stream>>>(qkv, g, E, ctx, lse, frames, axis);
    return cmgan_check_launch("attn_fwd_mma_kernel");
}

// tf32 tensor-core backward (same contract as cmgan_attention_bwd: dqkv overwritten, dE accumulated, delta scratch).
// parts: bit 0 = delta, bit 1 = dq + dE (reads delta), bit 2 = dk / dv (reads delta).  The two big kernels are independent of each other once
// delta exists and each one alone leaves most of an SM idle (8 - 12 resident warps, barrier- and latency-bound), so the caller may run
// part 1 first and then parts 2 and 4 on two streams; cmgan_attention_bwd_tf32 = all parts in order on one stream.
// scratch (optional, cmgan_attention_bwd_ws_floats): block-private dE accumulators in global memory -> the dq kernel needs 60 KB instead of
// 110+ KB of shared memory and runs 3 blocks / SM (any L) instead of 2 (1 at L = 1281).
static int dq_blocks(int ntile, int per_sm, int n_items) {
    int ng = (148 * per_sm) / ntile;
    if (ng < 1) ng = 1;
    return ng > n_items ? n_items : ng;
}

CMGAN_API long long cmgan_attention_bwd_ws_floats(int B, int T, int F, int axis) {
    if (axis != 0 && axis != 1) { cmgan_set_error("cmgan_attention_bwd_ws_floats: axis must be 0 (time) or 1 (freq)"); return -1; }
    SeqGeom g = make_seq_geom(B, T, F, axis);
    if (g.n_seq == 0 || g.L == 0) return 0;
    const int ntile = cdiv(g.L, QB), Lpad = ntile * KT;
    return (long long)dq_blocks(ntile, 3, g.n_seq * H) * ntile * (Lpad + 64) * D;
}

CMGAN_API int cmgan_attention_bwd_tf32_ws(const float* qkv, const float* E, const float* ctx, const float* dctx, const float* lse, int B,
                                          int T, int F, int axis, float* delta, float* dqkv, float* dE, int parts, float* scratch,
                                          long long scratch_floats, void* stream) {
    CMGAN_REQUIRE(qkv && E && ctx && dctx && lse && delta && dqkv && dE, "cmgan_attention_bwd_tf32: null pointer");
    CMGAN_REQUIRE(axis == 0 || axis == 1, "cmgan_attention_bwd_tf32: axis must be 0 (time) or 1 (freq)");
    SeqGeom g = make_seq_geom(B, T, F, axis);
    if (g.n_seq == 0 || g.L == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    const int ntile = cdiv(g.L, QB), Lpad = ntile * KT;
    const int n_items = g.n_seq * H;
    const bool gde = scratch != nullptr;
    if (gde) CMGAN_REQUIRE(scratch_floats >= cmgan_attention_bwd_ws_floats(B, T, F, axis) && (((uintptr_t)scratch) & 7) == 0,
                           "cmgan_attention_bwd_tf32_ws: scratch too small (%lld floats) or misaligned", scratch_floats);
    const int smem_dq = ((gde ? 1 : 2) * TILE_FLOATS + QB * LDRB + QB * LDS_ + (gde ? 0 : (Lpad + 64) * D)) * (int)sizeof(float);
    const int smem_kv = (2 * TILE_FLOATS + QB * LDR2 + 4 * QB) * (int)sizeof(float);
    CMGAN_REQUIRE(smem_dq <= 227 * 1024, "cmgan_attention_bwd_tf32: sequence length %d too long for the shared dE accumulator", g.L);
    static int smem_dq_set = 0;
    static bool kv_set = false, gde_set = false;
    if (!gde && smem_dq > smem_dq_set) {
        cudaError_t e = cudaFuncSetAttribute(attn_bwd_dq_mma_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_dq);
        CMGAN_REQUIRE(e == cudaSuccess, "cmgan_attention_bwd_tf32: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
        smem_dq_set = smem_dq;
    }
    if (gde && !gde_set) {
        cudaError_t e = cudaFuncSetAttribute(attn_bwd_dq_mma_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_dq);
        CMGAN_REQUIRE(e == cudaSuccess, "cmgan_attention_bwd_tf32: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
        gde_set = true;
    }
    if (!kv_set) {
        cudaError_t e = cudaFuncSetAttribute(attn_bwd_dkv_mma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_kv);
        CMGAN_REQUIRE(e == cudaSuccess, "cmgan_attention_bwd_tf32: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
        kv_set = true;
    }
    if (parts & 1) {
        const long n = (long)B * T * F * H;
        attn_delta_kernel<<<cdiv(n, 256), 256, 0, st>>>(ctx, dctx, n, delta);
        if (cmgan_check_launch("attn_delta_kernel")) return -1;
    }
    if (parts & 2) {
        if (gde)
            attn_bwd_dq_mma_kernel<true><<<dim3(dq_blocks(ntile, 3, n_items), ntile), 128, smem_dq, st>>>(qkv, g, E, ctx, dctx, lse, n_items, Lpad,
                                                                                                          delta, dqkv, dE, scratch);
        else
            attn_bwd_dq_mma_kernel<false><<<dim3(dq_blocks(ntile, 2, n_items), ntile), 128, smem_dq, st>>>(qkv, g, E, ctx, dctx, lse, n_items, Lpad,
                                                                                                           delta, dqkv, dE, nullptr);
        if (cmgan_check_launch("attn_bwd_dq_mma_kernel")) return -1;
    }
    if (parts & 4) {
        attn_bwd_dkv_mma_kernel<<<dim3(n_items, ntile), 128, smem_kv, st>>>(qkv, g, E, dctx, lse, delta, dqkv);
        if (cmgan_check_launch("attn_bwd_dkv_mma_kernel")) return -1;
    }
    return 0;
}

CMGAN_API int cmgan_attention_bwd_tf32_parts(const float* qkv, const float* E, const float* ctx, const float* dctx, const float* lse, int B,
                                             int T, int F, int axis, float* delta, float* dqkv, float* dE, int parts, void* stream) {
    return cmgan_attention_bwd_tf32_ws(qkv, E, ctx, dctx, lse, B, T, F, axis, delta, dqkv, dE, parts, nullptr, 0, stream);
}

CMGAN_API int cmgan_attention_bwd_tf32(const float* qkv, const float* E, const float* ctx, const float* dctx, const float* lse, int B,
                                       int T, int F, int axis, float* delta, float* dqkv, float* dE, void* stream) {
    return cmgan_attention_bwd_tf32_parts(qkv, E, ctx, dctx, lse, B, T, F, axis, delta, dqkv, dE, 7, stream);
}
