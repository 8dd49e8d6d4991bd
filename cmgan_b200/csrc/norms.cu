// LayerNorm / InstanceNorm / BatchNorm statistics, applies and gradients (HBM-bound row kernels).
// Channel-last rows; LayerNorm is over the 64 channels of one row (one warp per row, shuffle reductions);
// Instance/BatchNorm statistics are per (group, channel) over all rows of a group (group = batch element
// for InstanceNorm2d, a single group for BatchNorm1d), accumulated in double.
#include "common.cuh"
#include "../../include/cmgan_b200.h"

namespace {

constexpr int LN_C = 64;
constexpr float EPS = 1e-5f;

// ---------------------------------------------------------------- LayerNorm (ref: conformer.py:68,161,214)
// stats[m] = (mean, rstd)
__global__ void ln_stats_kernel(const float* __restrict__ x, long ldx, long M, float2* __restrict__ stats) {
    long row = (long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    int lane = threadIdx.x & 31;
    if (row >= M) return;
    float2 v = __ldg(reinterpret_cast<const float2*>(x + row * ldx) + lane);
    float mean = warp_sum(v.x + v.y) * (1.0f / LN_C);
    float d0 = v.x - mean, d1 = v.y - mean;
    float var = warp_sum(d0 * d0 + d1 * d1) * (1.0f / LN_C);
    if (lane == 0) stats[row] = make_float2(mean, rsqrtf(var + EPS));
}

// Both LayerNorm kernels: a row (64 channels) is held by HALF a warp as one float4 per lane, so every instruction covers two rows and a
// reduction is 4 shuffle steps; a warp walks LN_RPW consecutive rows with the per-channel parameters hoisted.  (The one-warp-per-row
// float2 form was issue-bound: 112 instructions per 256-byte row, 72 % issue-slot utilisation at 1.5 TB/s.)
constexpr int LN_RPW = 8;          // rows per warp (4 iterations of 2 rows)

__device__ __forceinline__ float half_warp_sum(float v) {
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// y = LN(x) * gamma + beta (+ res);  stats written for the backward pass
__global__ void __launch_bounds__(256) ln_apply_kernel(const float* __restrict__ x, long ldx, long M, const float* __restrict__ gamma,
                                                       const float* __restrict__ beta, const float* __restrict__ res, long ldr,
                                                       float* __restrict__ y, long ldy, float2* __restrict__ stats, int round_tf32) {
    const int lane = threadIdx.x & 31, hl = lane & 15, hw = lane >> 4;
    const long r0 = ((long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * LN_RPW + hw;
    const float4 g = __ldg(reinterpret_cast<const float4*>(gamma) + hl);
    const float4 b = __ldg(reinterpret_cast<const float4*>(beta) + hl);
#pragma unroll
    for (int it = 0; it < LN_RPW / 2; ++it) {
        const long row = r0 + 2 * it;
        const bool ok = row < M;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f), r = v;
        if (ok) {
            v = __ldg(reinterpret_cast<const float4*>(x + row * ldx) + hl);
            if (res) r = __ldg(reinterpret_cast<const float4*>(res + row * ldr) + hl);
        }
        const float mean = half_warp_sum((v.x + v.y) + (v.z + v.w)) * (1.0f / LN_C);
        const float d0 = v.x - mean, d1 = v.y - mean, d2 = v.z - mean, d3 = v.w - mean;
        const float var = half_warp_sum((d0 * d0 + d1 * d1) + (d2 * d2 + d3 * d3)) * (1.0f / LN_C);
        const float rstd = rsqrtf(var + EPS);
        float4 o = make_float4(fmaf(d0 * rstd, g.x, b.x) + r.x, fmaf(d1 * rstd, g.y, b.y) + r.y, fmaf(d2 * rstd, g.z, b.z) + r.z,
                               fmaf(d3 * rstd, g.w, b.w) + r.w);
        if (round_tf32) {      // consumer is a tf32 tensor-core GEMM fed by TMA / cp.async: round (not truncate) once, here
            o.x = cmgan_rna_tf32(o.x); o.y = cmgan_rna_tf32(o.y); o.z = cmgan_rna_tf32(o.z); o.w = cmgan_rna_tf32(o.w);
        }
        if (ok) {
            reinterpret_cast<float4*>(y + row * ldy)[hl] = o;
            if (stats && hl == 0) stats[row] = make_float2(mean, rstd);
        }
    }
}

// dx = rstd * (dy*g - mean(dy*g) - xhat * mean(dy*g*xhat)) (+ res);  dgamma += sum dy*xhat;  dbeta += sum dy
__global__ void __launch_bounds__(256) ln_bwd_kernel(const float* __restrict__ dy, long lddy, const float* __restrict__ x, long ldx,
                              const float2* __restrict__ stats, const float* __restrict__ gamma, long M,
                              const float* __restrict__ res, long ldr, const float* __restrict__ res2, long ldr2,
                              float* __restrict__ dx, long lddx,
                              float* __restrict__ dgamma, float* __restrict__ dbeta, int rows_per_warp,
                              float* __restrict__ dz, long lddz, float zalpha, unsigned long long zseed, unsigned zthr, float zinv_keep,
                              const unsigned long long* __restrict__ seed_dev, int rnd) {
    __shared__ float4 sg[16][LN_C / 4], sb[16][LN_C / 4];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, hl = lane & 15, hw = lane >> 4, nw = blockDim.x >> 5;
    const long r0 = ((long)blockIdx.x * nw + warp) * rows_per_warp + hw;
    const float4 g = __ldg(reinterpret_cast<const float4*>(gamma) + hl);
    float4 ag = make_float4(0.f, 0.f, 0.f, 0.f), ab = ag;
    // optional second output dz = zalpha * dropmask(zseed) * dx: the gradient entering the next residual branch, whose forward output
    // went through dropout (mask regenerated from the element index row * 64 + channel, as in the GEMM epilogue that applied it)
    const uint32_t zs32 = dz ? cmgan_seed32(cmgan_eff_seed(zseed, seed_dev)) : 0u;
    const uint32_t zt16 = zthr >> 16;
    const float zk = zalpha * zinv_keep;
    for (int i = 0; i < rows_per_warp; i += 2) {
        const long row = r0 + i;
        const bool ok = row < M;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f), d = v, r = v;
        float2 st = make_float2(0.f, 0.f);
        if (ok) {
            v = __ldg(reinterpret_cast<const float4*>(x + row * ldx) + hl);
            d = __ldg(reinterpret_cast<const float4*>(dy + row * lddy) + hl);
            st = __ldg(stats + row);
            if (res) r = __ldg(reinterpret_cast<const float4*>(res + row * ldr) + hl);
            if (res2) {
                const float4 r2 = __ldg(reinterpret_cast<const float4*>(res2 + row * ldr2) + hl);
                r.x += r2.x; r.y += r2.y; r.z += r2.z; r.w += r2.w;
            }
        }
        const float xh0 = (v.x - st.x) * st.y, xh1 = (v.y - st.x) * st.y, xh2 = (v.z - st.x) * st.y, xh3 = (v.w - st.x) * st.y;
        const float dg0 = d.x * g.x, dg1 = d.y * g.y, dg2 = d.z * g.z, dg3 = d.w * g.w;
        const float m1 = half_warp_sum((dg0 + dg1) + (dg2 + dg3)) * (1.0f / LN_C);
        const float m2 = half_warp_sum((dg0 * xh0 + dg1 * xh1) + (dg2 * xh2 + dg3 * xh3)) * (1.0f / LN_C);
        const float4 o = make_float4(st.y * (dg0 - m1 - xh0 * m2) + r.x, st.y * (dg1 - m1 - xh1 * m2) + r.y,
                                     st.y * (dg2 - m1 - xh2 * m2) + r.z, st.y * (dg3 - m1 - xh3 * m2) + r.w);
        if (ok) {
            reinterpret_cast<float4*>(dx + row * lddx)[hl] = o;
            if (dz) {
                float s0 = zalpha, s1 = zalpha, s2 = zalpha, s3 = zalpha;
                if (zthr) {          // one hash per pair of channels (2 p, 2 p + 1), pair index = row * 32 + p
                    const uint32_t h0 = cmgan_pair_hash(zs32, (uint64_t)row * (LN_C / 2) + 2 * hl);
                    const uint32_t h1 = cmgan_pair_hash(zs32, (uint64_t)row * (LN_C / 2) + 2 * hl + 1);
                    s0 = (h0 & 0xFFFFu) >= zt16 ? zk : 0.f; s1 = (h0 >> 16) >= zt16 ? zk : 0.f;
                    s2 = (h1 & 0xFFFFu) >= zt16 ? zk : 0.f; s3 = (h1 >> 16) >= zt16 ? zk : 0.f;
                }
                reinterpret_cast<float4*>(dz + row * lddz)[hl] = make_float4(cmgan_maybe_rna(o.x * s0, rnd), cmgan_maybe_rna(o.y * s1, rnd),
                                                                             cmgan_maybe_rna(o.z * s2, rnd), cmgan_maybe_rna(o.w * s3, rnd));
            }
        }
        ag.x = fmaf(d.x, xh0, ag.x); ag.y = fmaf(d.y, xh1, ag.y); ag.z = fmaf(d.z, xh2, ag.z); ag.w = fmaf(d.w, xh3, ag.w);
        ab.x += d.x; ab.y += d.y; ab.z += d.z; ab.w += d.w;
    }
    sg[warp * 2 + hw][hl] = ag;
    sb[warp * 2 + hw][hl] = ab;
    __syncthreads();
    if (threadIdx.x < LN_C) {
        float a = 0.f, b = 0.f;
        for (int w = 0; w < 2 * nw; ++w) { a += reinterpret_cast<const float*>(sg[w])[threadIdx.x]; b += reinterpret_cast<const float*>(sb[w])[threadIdx.x]; }
        atomicAdd(dgamma + threadIdx.x, a);
        atomicAdd(dbeta + threadIdx.x, b);
    }
}

// ---------------------------------------------------------------- group statistics (InstanceNorm2d / BatchNorm1d)
// sums[(grp*C + c)*2 + {0,1}] += sum x, sum x^2 over the rows of group grp.  Block = one chunk of rows of
// one group; thread = (row-subgroup, channel).  frames (optional, ragged batch): group grp covers its first frames[grp] * rows_per_frame
// rows only (the rows of padded frames are never read).
template <bool VAR>
__device__ __forceinline__ long group_rows(long rows_per_group, const int* __restrict__ frames, long rows_per_frame, int grp) {
    return VAR ? (long)varlen_frames(frames, grp, (int)(rows_per_group / rows_per_frame)) * rows_per_frame : rows_per_group;
}

template <bool VAR>
__global__ void norm_stats_kernel(const float* __restrict__ x, long ldx, long rows_per_group, int C, int chunk,
                                  double* __restrict__ sums, const int* __restrict__ frames, long rows_per_frame) {
    extern __shared__ double sm[];
    int grp = blockIdx.y;
    const long rows = group_rows<VAR>(rows_per_group, frames, rows_per_frame, grp);
    long r_beg = (long)blockIdx.x * chunk;
    if (VAR && r_beg >= rows) return;
    long r_end = r_beg + chunk < rows ? r_beg + chunk : rows;
    int c = threadIdx.x % C, rg = threadIdx.x / C, nrg = blockDim.x / C;
    float s = 0.f, q = 0.f;
    const float* base = x + ((long)grp * rows_per_group) * ldx + c;
    if (rg < nrg)
        for (long r = r_beg + rg; r < r_end; r += nrg) { float v = __ldg(base + r * ldx); s += v; q = fmaf(v, v, q); }
    sm[threadIdx.x * 2] = s; sm[threadIdx.x * 2 + 1] = q;
    __syncthreads();
    if (threadIdx.x < C) {
        double ds = 0.0, dq = 0.0;
        for (int g = 0; g < nrg; ++g) { ds += sm[(g * C + c) * 2]; dq += sm[(g * C + c) * 2 + 1]; }
        atomicAdd(sums + ((long)grp * C + c) * 2, ds);
        atomicAdd(sums + ((long)grp * C + c) * 2 + 1, dq);
    }
}

// same, 128-bit loads: thread = (row-subgroup, 4 channels); C, ldx multiples of 4, x 16-byte aligned
template <bool VAR>
__global__ void norm_stats4_kernel(const float* __restrict__ x, long ldx, long rows_per_group, int C, int chunk, double* __restrict__ sums,
                                   const int* __restrict__ frames, long rows_per_frame) {
    __shared__ float sm[256][8];
    const int grp = blockIdx.y, cv = C / 4;
    const long rows = group_rows<VAR>(rows_per_group, frames, rows_per_frame, grp);
    const long r_beg = (long)blockIdx.x * chunk;
    if (VAR && r_beg >= rows) return;
    const long r_end = r_beg + chunk < rows ? r_beg + chunk : rows;
    const int c4 = threadIdx.x % cv, rg = threadIdx.x / cv, nrg = blockDim.x / cv;
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f), q = s;
    const float* base = x + ((long)grp * rows_per_group) * ldx + c4 * 4;
    if (rg < nrg) {
#pragma unroll 4
        for (long r = r_beg + rg; r < r_end; r += nrg) {
            const float4 v = __ldg(reinterpret_cast<const float4*>(base + r * ldx));
            s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
            q.x = fmaf(v.x, v.x, q.x); q.y = fmaf(v.y, v.y, q.y); q.z = fmaf(v.z, v.z, q.z); q.w = fmaf(v.w, v.w, q.w);
        }
    }
    float* o = sm[threadIdx.x];
    o[0] = s.x; o[1] = s.y; o[2] = s.z; o[3] = s.w; o[4] = q.x; o[5] = q.y; o[6] = q.z; o[7] = q.w;
    __syncthreads();
    if (threadIdx.x < C) {
        const int c = threadIdx.x, cc = c >> 2, j = c & 3;
        double ds = 0.0, dq = 0.0;
        for (int g = 0; g < nrg; ++g) { ds += sm[g * cv + cc][j]; dq += sm[g * cv + cc][4 + j]; }
        atomicAdd(sums + ((long)grp * C + c) * 2, ds);
        atomicAdd(sums + ((long)grp * C + c) * 2 + 1, dq);
    }
}

// mode 0: InstanceNorm / train-mode BatchNorm: statistics from sums (biased variance for the normalisation)
// mode 1: eval-mode BatchNorm: running statistics
// outputs per (grp, c): scale = gamma*rstd, shift = beta - mean*scale, mean, rstd (table stride = tstride)
// when running_mean != null and mode 0: running <- (1-mom)*running + mom*(mean, unbiased var) (BatchNorm1d train)
// frames (optional, mode 0, ragged batch): group grp averages over n_g = frames[grp] * n rows (n = rows per frame, frames[grp] <= T)
__global__ void norm_finalize_kernel(const double* __restrict__ sums, long n, int G, int C, int mode,
                                     const float* __restrict__ gamma, const float* __restrict__ beta,
                                     float* __restrict__ running_mean, float* __restrict__ running_var, float momentum,
                                     float* __restrict__ scale, float* __restrict__ shift, float* __restrict__ mean_out,
                                     float* __restrict__ rstd_out, long tstride, const int* __restrict__ frames, int T) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= G * C) return;
    int grp = i / C, c = i % C;
    if (frames) n *= varlen_frames(frames, grp, T);
    float mean, var;
    if (mode == 1) { mean = running_mean[c]; var = running_var[c]; }
    else {
        double m = sums[(long)i * 2] / (double)n;
        double v = sums[(long)i * 2 + 1] / (double)n - m * m;
        if (v < 0.0) v = 0.0;
        mean = (float)m; var = (float)v;
        if (running_mean) {
            double unb = n > 1 ? v * (double)n / (double)(n - 1) : v;
            running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * mean;
            running_var[c] = (1.f - momentum) * running_var[c] + momentum * (float)unb;
        }
    }
    float rstd = rsqrtf(var + EPS);
    float sc = gamma[c] * rstd;
    long o = (long)grp * tstride + c;
    scale[o] = sc; shift[o] = beta[c] - mean * sc;
    if (mean_out) mean_out[o] = mean;
    if (rstd_out) rstd_out[o] = rstd;
}

// backward pass 1.  z = x*scale + shift; act: 0 none, 1 PReLU(slope[c]);  g = dact * act'(z)
//   S[(grp*C+c)*2 + {0,1}] += sum g, sum g*xhat   (xhat = (x - mean) * rstd);   dslope[c] += sum dact * z * [z<0]
__global__ void norm_bwd_reduce_kernel(const float* __restrict__ x, long ldx, const float* __restrict__ dact, long ldd,
                                       long rows_per_group, int C, int chunk, int act, const float* __restrict__ scale,
                                       const float* __restrict__ shift, const float* __restrict__ mean,
                                       const float* __restrict__ rstd, long tstride, const float* __restrict__ slope,
                                       double* __restrict__ S, float* __restrict__ dslope) {
    extern __shared__ double sm[];
    int grp = blockIdx.y;
    long r_beg = (long)blockIdx.x * chunk;
    long r_end = r_beg + chunk < rows_per_group ? r_beg + chunk : rows_per_group;
    int c = threadIdx.x % C, rg = threadIdx.x / C, nrg = blockDim.x / C;
    float s1 = 0.f, s2 = 0.f, s3 = 0.f;
    if (rg < nrg) {
        long t = (long)grp * tstride + c;
        float sc = scale[t], sh = shift[t], mu = mean[t], rs = rstd[t];
        float a = act ? slope[c] : 1.f;
        long rb = (long)grp * rows_per_group;
        for (long r = r_beg + rg; r < r_end; r += nrg) {
            float v = __ldg(x + (rb + r) * ldx + c);
            float d = __ldg(dact + (rb + r) * ldd + c);
            float z = v * sc + sh;
            float gq = d;
            if (act && z < 0.f) { gq = d * a; s3 = fmaf(d, z, s3); }
            s1 += gq; s2 = fmaf(gq, (v - mu) * rs, s2);
        }
    }
    sm[threadIdx.x * 3] = s1; sm[threadIdx.x * 3 + 1] = s2; sm[threadIdx.x * 3 + 2] = s3;
    __syncthreads();
    if (threadIdx.x < C) {
        double a1 = 0, a2 = 0, a3 = 0;
        for (int g = 0; g < nrg; ++g) { a1 += sm[(g * C + c) * 3]; a2 += sm[(g * C + c) * 3 + 1]; a3 += sm[(g * C + c) * 3 + 2]; }
        atomicAdd(S + ((long)grp * C + c) * 2, a1);
        atomicAdd(S + ((long)grp * C + c) * 2 + 1, a2);
        if (act && dslope) atomicAdd(dslope + c, (float)a3);
    }
}

// same, 128-bit loads: thread = (row-subgroup, 4 channels); C, ldx, ldd, tstride multiples of 4, 16-byte aligned pointers
__global__ void norm_bwd_reduce4_kernel(const float* __restrict__ x, long ldx, const float* __restrict__ dact, long ldd,
                                        long rows_per_group, int C, int chunk, int act, const float* __restrict__ scale,
                                        const float* __restrict__ shift, const float* __restrict__ mean,
                                        const float* __restrict__ rstd, long tstride, const float* __restrict__ slope,
                                        double* __restrict__ S, float* __restrict__ dslope) {
    __shared__ float sm[256][12];
    const int grp = blockIdx.y, cv = C / 4;
    const long r_beg = (long)blockIdx.x * chunk;
    const long r_end = r_beg + chunk < rows_per_group ? r_beg + chunk : rows_per_group;
    const int c4 = threadIdx.x % cv, rg = threadIdx.x / cv, nrg = blockDim.x / cv;
    float s1[4] = {0.f, 0.f, 0.f, 0.f}, s2[4] = {0.f, 0.f, 0.f, 0.f}, s3[4] = {0.f, 0.f, 0.f, 0.f};
    if (rg < nrg) {
        const long t = (long)grp * tstride + c4 * 4;
        const float4 sc4 = __ldg(reinterpret_cast<const float4*>(scale + t)), sh4 = __ldg(reinterpret_cast<const float4*>(shift + t));
        const float4 mu4 = __ldg(reinterpret_cast<const float4*>(mean + t)), rs4 = __ldg(reinterpret_cast<const float4*>(rstd + t));
        float4 a4 = make_float4(1.f, 1.f, 1.f, 1.f);
        if (act) a4 = __ldg(reinterpret_cast<const float4*>(slope + c4 * 4));
        const float sc[4] = {sc4.x, sc4.y, sc4.z, sc4.w}, sh[4] = {sh4.x, sh4.y, sh4.z, sh4.w}, mu[4] = {mu4.x, mu4.y, mu4.z, mu4.w};
        const float rs[4] = {rs4.x, rs4.y, rs4.z, rs4.w}, a[4] = {a4.x, a4.y, a4.z, a4.w};
        const long rb = (long)grp * rows_per_group;
#pragma unroll 4
        for (long r = r_beg + rg; r < r_end; r += nrg) {
            const float4 v4 = __ldg(reinterpret_cast<const float4*>(x + (rb + r) * ldx) + c4);
            const float4 d4 = __ldg(reinterpret_cast<const float4*>(dact + (rb + r) * ldd) + c4);
            const float v[4] = {v4.x, v4.y, v4.z, v4.w}, d[4] = {d4.x, d4.y, d4.z, d4.w};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float z = fmaf(v[j], sc[j], sh[j]);
                float gq = d[j];
                if (act && z < 0.f) { gq = d[j] * a[j]; s3[j] = fmaf(d[j], z, s3[j]); }
                s1[j] += gq; s2[j] = fmaf(gq, (v[j] - mu[j]) * rs[j], s2[j]);
            }
        }
    }
    float* o = sm[threadIdx.x];
#pragma unroll
    for (int j = 0; j < 4; ++j) { o[j] = s1[j]; o[4 + j] = s2[j]; o[8 + j] = s3[j]; }
    __syncthreads();
    if (threadIdx.x < C) {
        const int c = threadIdx.x, cc = c >> 2, j = c & 3;
        double a1 = 0, a2 = 0, a3 = 0;
        for (int g = 0; g < nrg; ++g) { a1 += sm[g * cv + cc][j]; a2 += sm[g * cv + cc][4 + j]; a3 += sm[g * cv + cc][8 + j]; }
        atomicAdd(S + ((long)grp * C + c) * 2, a1);
        atomicAdd(S + ((long)grp * C + c) * 2 + 1, a2);
        if (act && dslope) atomicAdd(dslope + c, (float)a3);
    }
}

// backward pass 2.  dx = scale * (g - [train] (S1/n + xhat*S2/n));  also dgamma[c] += S2, dbeta[c] += S1 (first chunk of each group)
// Block = one chunk of rows of one group; thread = (row-subgroup, channel): the per-(group, channel) constants are loaded once.
__global__ void norm_bwd_apply_kernel(const float* __restrict__ x, long ldx, const float* __restrict__ dact, long ldd,
                                      long rows_per_group, int C, int chunk, int act, int use_batch_stats,
                                      const float* __restrict__ scale, const float* __restrict__ shift,
                                      const float* __restrict__ mean, const float* __restrict__ rstd, long tstride,
                                      const float* __restrict__ slope, const double* __restrict__ S,
                                      float* __restrict__ dx, long lddx, float* __restrict__ dgamma, float* __restrict__ dbeta, int rnd) {
    const int grp = blockIdx.y;
    const long r_beg = (long)blockIdx.x * chunk;
    const long r_end = r_beg + chunk < rows_per_group ? r_beg + chunk : rows_per_group;
    const int c = threadIdx.x % C, rg = threadIdx.x / C, nrg = blockDim.x / C;
    if (rg >= nrg) return;
    const long t = (long)grp * tstride + c;
    const float sc = scale[t], sh = shift[t], mu = mean[t], rs = rstd[t];
    const float a = act ? slope[c] : 1.f;
    const double s1 = S[((long)grp * C + c) * 2], s2 = S[((long)grp * C + c) * 2 + 1];
    if (blockIdx.x == 0 && rg == 0 && dgamma) { atomicAdd(dgamma + c, (float)s2); atomicAdd(dbeta + c, (float)s1); }
    float m1 = 0.f, m2 = 0.f;
    if (use_batch_stats) { m1 = (float)(s1 / (double)rows_per_group); m2 = (float)(s2 / (double)rows_per_group); }
    const long rb = (long)grp * rows_per_group;
    for (long r = r_beg + rg; r < r_end; r += nrg) {
        const float v = __ldg(x + (rb + r) * ldx + c), d = __ldg(dact + (rb + r) * ldd + c);
        const float z = v * sc + sh;
        const float gq = (act && z < 0.f) ? d * a : d;
        dx[(rb + r) * lddx + c] = cmgan_maybe_rna(sc * (gq - m1 - (v - mu) * rs * m2), rnd);
    }
}

// same, 128-bit accesses: thread = (row-subgroup, 4 channels)
__global__ void norm_bwd_apply4_kernel(const float* __restrict__ x, long ldx, const float* __restrict__ dact, long ldd,
                                       long rows_per_group, int C, int chunk, int act, int use_batch_stats,
                                       const float* __restrict__ scale, const float* __restrict__ shift,
                                       const float* __restrict__ mean, const float* __restrict__ rstd, long tstride,
                                       const float* __restrict__ slope, const double* __restrict__ S,
                                       float* __restrict__ dx, long lddx, float* __restrict__ dgamma, float* __restrict__ dbeta, int rnd) {
    const int grp = blockIdx.y, cv = C / 4;
    const long r_beg = (long)blockIdx.x * chunk;
    const long r_end = r_beg + chunk < rows_per_group ? r_beg + chunk : rows_per_group;
    const int c4 = threadIdx.x % cv, rg = threadIdx.x / cv, nrg = blockDim.x / cv;
    if (rg >= nrg) return;
    const long t = (long)grp * tstride + c4 * 4;
    const float4 sc4 = __ldg(reinterpret_cast<const float4*>(scale + t)), sh4 = __ldg(reinterpret_cast<const float4*>(shift + t));
    const float4 mu4 = __ldg(reinterpret_cast<const float4*>(mean + t)), rs4 = __ldg(reinterpret_cast<const float4*>(rstd + t));
    float4 a4 = make_float4(1.f, 1.f, 1.f, 1.f);
    if (act) a4 = __ldg(reinterpret_cast<const float4*>(slope + c4 * 4));
    const float sc[4] = {sc4.x, sc4.y, sc4.z, sc4.w}, sh[4] = {sh4.x, sh4.y, sh4.z, sh4.w}, mu[4] = {mu4.x, mu4.y, mu4.z, mu4.w};
    const float rs[4] = {rs4.x, rs4.y, rs4.z, rs4.w}, a[4] = {a4.x, a4.y, a4.z, a4.w};
    float m1[4], m2[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int c = c4 * 4 + j;
        const double s1 = S[((long)grp * C + c) * 2], s2 = S[((long)grp * C + c) * 2 + 1];
        if (blockIdx.x == 0 && rg == 0 && dgamma) { atomicAdd(dgamma + c, (float)s2); atomicAdd(dbeta + c, (float)s1); }
        m1[j] = use_batch_stats ? (float)(s1 / (double)rows_per_group) : 0.f;
        m2[j] = use_batch_stats ? (float)(s2 / (double)rows_per_group) : 0.f;
    }
    const long rb = (long)grp * rows_per_group;
#pragma unroll 4
    for (long r = r_beg + rg; r < r_end; r += nrg) {
        const float4 v4 = __ldg(reinterpret_cast<const float4*>(x + (rb + r) * ldx) + c4);
        const float4 d4 = __ldg(reinterpret_cast<const float4*>(dact + (rb + r) * ldd) + c4);
        const float v[4] = {v4.x, v4.y, v4.z, v4.w}, d[4] = {d4.x, d4.y, d4.z, d4.w};
        float o[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const float z = fmaf(v[j], sc[j], sh[j]);
            const float gq = (act && z < 0.f) ? d[j] * a[j] : d[j];
            o[j] = cmgan_maybe_rna(sc[j] * (gq - m1[j] - (v[j] - mu[j]) * rs[j] * m2[j]), rnd);
        }
        *reinterpret_cast<float4*>(dx + (rb + r) * lddx + c4 * 4) = make_float4(o[0], o[1], o[2], o[3]);
    }
}

// y[row, c] = act(x*scale+shift) materialised (used where the consumer is not a GEMM with a prologue)
__device__ __forceinline__ float norm_act1(float z, int a, float sl, bool round_tf32) {
    if (a == 1 && z < 0.f) z *= sl;
    else if (a == 2) z = swishf_(z);
    if (round_tf32) {      // consumer is a tf32 tensor-core GEMM fed by cp.async / TMA: round (not truncate) once, here
        uint32_t r;
        asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(z));
        z = __uint_as_float(r);
    }
    return z;
}
// VEC = 4: C, ldx, ldy, tstride multiples of 4 and 16-byte aligned pointers (every call of the hot path); VEC = 1: general
template <int VEC>
__global__ void norm_apply_kernel(const float* __restrict__ x, long ldx, long rows_per_group, int G, int C, int act,
                                  const float* __restrict__ scale, const float* __restrict__ shift, long tstride,
                                  const float* __restrict__ slope, float* __restrict__ y, long ldy) {
    const int cv = C / VEC;
    long total = (long)G * rows_per_group * cv;
    long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    int c = (int)(i % cv) * VEC;
    long row = i / cv;
    long t = (row / rows_per_group) * tstride + c;
    const int a = act & 15;
    const bool rnd = (act & 16) != 0;
    if (VEC == 4) {
        const float4 v = __ldg(reinterpret_cast<const float4*>(x + row * ldx + c));
        const float4 sc = __ldg(reinterpret_cast<const float4*>(scale + t)), sh = __ldg(reinterpret_cast<const float4*>(shift + t));
        float4 sl = make_float4(0.f, 0.f, 0.f, 0.f);
        if (a == 1) sl = __ldg(reinterpret_cast<const float4*>(slope + c));
        float4 o;
        o.x = norm_act1(fmaf(v.x, sc.x, sh.x), a, sl.x, rnd); o.y = norm_act1(fmaf(v.y, sc.y, sh.y), a, sl.y, rnd);
        o.z = norm_act1(fmaf(v.z, sc.z, sh.z), a, sl.z, rnd); o.w = norm_act1(fmaf(v.w, sc.w, sh.w), a, sl.w, rnd);
        *reinterpret_cast<float4*>(y + row * ldy + c) = o;
    } else {
        float z = fmaf(__ldg(x + row * ldx + c), scale[t], shift[t]);
        y[row * ldy + c] = norm_act1(z, a, a == 1 ? slope[c] : 0.f, rnd);
    }
}

__global__ void fill_kernel(float* p, long n, float v) {
    long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}
__global__ void copy_rows_kernel(const float* __restrict__ src, long lds, float* __restrict__ dst, long ldd, long M, int C, int rnd) {
    long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    long total = M * (C / 4);
    if (i >= total) return;
    long row = i / (C / 4); int c4 = (int)(i % (C / 4));
    float4 v = __ldg(reinterpret_cast<const float4*>(src + row * lds) + c4);
    if (rnd) v = make_float4(cmgan_rna_tf32(v.x), cmgan_rna_tf32(v.y), cmgan_rna_tf32(v.z), cmgan_rna_tf32(v.w));
    reinterpret_cast<float4*>(dst + row * ldd)[c4] = v;
}

__global__ void add_rows_kernel(const float* __restrict__ src, long lds, float* __restrict__ dst, long ldd, long M, int C) {
    long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    long total = M * (C / 4);
    if (i >= total) return;
    long row = i / (C / 4); int c4 = (int)(i % (C / 4));
    float4 a = __ldg(reinterpret_cast<const float4*>(src + row * lds) + c4);
    float4* d = reinterpret_cast<float4*>(dst + row * ldd) + c4;
    float4 b = *d;
    *d = make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w);
}

}  // namespace

CMGAN_API int cmgan_ln_stats(const float* x, long long ldx, long long M, float* stats, void* stream) {
    CMGAN_REQUIRE(x && stats && ldx % 2 == 0, "cmgan_ln_stats: bad arguments");
    if (M == 0) return 0;
    ln_stats_kernel<<<cdiv(M, 8), 256, 0, (cudaStream_t)stream>>>(x, ldx, M, reinterpret_cast<float2*>(stats));
    return cmgan_check_launch("ln_stats_kernel");
}

// y = LayerNorm(x) * gamma + beta + res  (res, stats optional); reference conformer.py:214,222 + generator.py:95,97
CMGAN_API int cmgan_ln_apply(const float* x, long long ldx, long long M, const float* gamma, const float* beta,
                             const float* res, long long ldr, float* y, long long ldy, float* stats, int round_tf32, void* stream) {
    CMGAN_REQUIRE(x && y && gamma && beta && ldx % 4 == 0 && ldy % 4 == 0 && ldr % 4 == 0 &&
                  ((((uintptr_t)x) | ((uintptr_t)y) | ((uintptr_t)res) | ((uintptr_t)gamma) | ((uintptr_t)beta)) & 15) == 0,
                  "cmgan_ln_apply: pointers must be 16-byte aligned, leading dimensions multiples of 4");
    if (M == 0) return 0;
    ln_apply_kernel<<<cdiv(M, 8 * LN_RPW), 256, 0, (cudaStream_t)stream>>>(x, ldx, M, gamma, beta, res, ldr, y, ldy,
                                                                 reinterpret_cast<float2*>(stats), round_tf32);
    return cmgan_check_launch("ln_apply_kernel");
}

static int ln_bwd_launch(const float* dy, long long lddy, const float* x, long long ldx, const float* stats, const float* gamma, long long M,
                         const float* res, long long ldr, const float* res2, long long ldr2, float* dx, long long lddx, float* dgamma,
                         float* dbeta, float* dz, long long lddz, float zalpha, unsigned long long zseed, unsigned zthr, float zinv_keep,
                         const unsigned long long* seed_dev, void* stream, const char* who) {
    CMGAN_REQUIRE(dy && x && stats && gamma && dx && dgamma && dbeta, "%s: null pointer", who);
    CMGAN_REQUIRE(lddy % 4 == 0 && ldx % 4 == 0 && lddx % 4 == 0 && ldr % 4 == 0 && ldr2 % 4 == 0 && lddz % 4 == 0 &&
                  ((((uintptr_t)dy) | ((uintptr_t)x) | ((uintptr_t)dx) | ((uintptr_t)res) | ((uintptr_t)res2) | ((uintptr_t)dz) | ((uintptr_t)gamma)) & 15) == 0,
                  "%s: pointers must be 16-byte aligned, leading dimensions multiples of 4", who);
    if (M == 0) return 0;
    const int rpw = 16;
    ln_bwd_kernel<<<cdiv(M, 8 * rpw), 256, 0, (cudaStream_t)stream>>>(dy, lddy, x, ldx, reinterpret_cast<const float2*>(stats), gamma, M, res, ldr,
                                                                     res2, ldr2, dx, lddx, dgamma, dbeta, rpw, dz, lddz, zalpha, zseed, zthr,
                                                                     zinv_keep, seed_dev, g_cmgan_round_tf32);
    return cmgan_check_launch("ln_bwd_kernel");
}

CMGAN_API int cmgan_ln_bwd(const float* dy, long long lddy, const float* x, long long ldx, const float* stats,
                           const float* gamma, long long M, const float* res, long long ldr, const float* res2, long long ldr2,
                           float* dx, long long lddx, float* dgamma, float* dbeta, void* stream) {
    return ln_bwd_launch(dy, lddy, x, ldx, stats, gamma, M, res, ldr, res2, ldr2, dx, lddx, dgamma, dbeta, nullptr, 0, 1.f, 0ull, 0u, 1.f, nullptr,
                         stream, "cmgan_ln_bwd");
}

// same, plus dz = alpha * dropout_scale(seed; element index row * 64 + c) * dx  (thr = p * 2^32, 0 = no dropout)
CMGAN_API int cmgan_ln_bwd_drop(const float* dy, long long lddy, const float* x, long long ldx, const float* stats, const float* gamma,
                                long long M, const float* res, long long ldr, const float* res2, long long ldr2, float* dx, long long lddx,
                                float* dgamma, float* dbeta, float* dz, long long lddz, float alpha, unsigned long long seed, unsigned int thr,
                                float inv_keep, const unsigned long long* seed_dev, void* stream) {
    CMGAN_REQUIRE(dz != nullptr, "cmgan_ln_bwd_drop: dz is null");
    return ln_bwd_launch(dy, lddy, x, ldx, stats, gamma, M, res, ldr, res2, ldr2, dx, lddx, dgamma, dbeta, dz, lddz, alpha, seed, thr, inv_keep,
                         seed_dev, stream, "cmgan_ln_bwd_drop");
}

static int norm_threads(int C) { return C <= 256 ? 256 : C; }

// sums must be zeroed by the caller (G*C*2 doubles).
static int norm_stats_launch(const float* x, long long ldx, int G, long long rows_per_group, int C, const int* frames, long long rows_per_frame,
                             double* sums, void* stream) {
    CMGAN_REQUIRE(x && sums && C >= 1 && C <= 256 && 256 % C == 0, "cmgan_norm_stats: C=%d unsupported", C);
    if (G == 0 || rows_per_group == 0) return 0;
    if (C % 4 == 0 && ldx % 4 == 0 && (((uintptr_t)x) & 15) == 0) {
        const int nrg4 = 256 / (C / 4);
        const int chunk4 = nrg4 * 16;                 // 16 x 128-bit loads per thread; ~1000 blocks on the hot shapes
        dim3 grid4(cdiv(rows_per_group, chunk4), G);
        if (frames) norm_stats4_kernel<true><<<grid4, 256, 0, (cudaStream_t)stream>>>(x, ldx, rows_per_group, C, chunk4, sums, frames, rows_per_frame);
        else norm_stats4_kernel<false><<<grid4, 256, 0, (cudaStream_t)stream>>>(x, ldx, rows_per_group, C, chunk4, sums, nullptr, 1);
        return cmgan_check_launch("norm_stats4_kernel");
    }
    int nrg = 256 / C;
    int chunk = nrg * 64;
    dim3 grid(cdiv(rows_per_group, chunk), G);
    const size_t smem = 256 * 2 * sizeof(double);
    if (frames) norm_stats_kernel<true><<<grid, norm_threads(C), smem, (cudaStream_t)stream>>>(x, ldx, rows_per_group, C, chunk, sums, frames, rows_per_frame);
    else norm_stats_kernel<false><<<grid, norm_threads(C), smem, (cudaStream_t)stream>>>(x, ldx, rows_per_group, C, chunk, sums, nullptr, 1);
    return cmgan_check_launch("norm_stats_kernel");
}

CMGAN_API int cmgan_norm_stats(const float* x, long long ldx, int G, long long rows_per_group, int C, double* sums, void* stream) {
    return norm_stats_launch(x, ldx, G, rows_per_group, C, nullptr, 1, sums, stream);
}

// ragged batch: group g (stride rows_per_group = T * rows_per_frame) covers its first frames[g] * rows_per_frame rows
CMGAN_API int cmgan_norm_stats_varlen(const float* x, long long ldx, int G, long long rows_per_group, int C, const int* frames,
                                      long long rows_per_frame, double* sums, void* stream) {
    CMGAN_REQUIRE(frames && rows_per_frame > 0 && rows_per_group % rows_per_frame == 0,
                  "cmgan_norm_stats_varlen: rows_per_group must be a multiple of rows_per_frame > 0");
    return norm_stats_launch(x, ldx, G, rows_per_group, C, frames, rows_per_frame, sums, stream);
}

CMGAN_API int cmgan_norm_finalize(const double* sums, long long n, int G, int C, int mode, const float* gamma, const float* beta,
                                  float* running_mean, float* running_var, float momentum, float* scale, float* shift,
                                  float* mean_out, float* rstd_out, long long tstride, void* stream) {
    CMGAN_REQUIRE(gamma && beta && scale && shift, "cmgan_norm_finalize: null pointer");
    CMGAN_REQUIRE(mode == 1 ? (running_mean && running_var) : (sums != nullptr), "cmgan_norm_finalize: missing statistics");
    norm_finalize_kernel<<<cdiv((long)G * C, 128), 128, 0, (cudaStream_t)stream>>>(sums, n, G, C, mode, gamma, beta, running_mean,
                                                                                 running_var, momentum, scale, shift, mean_out,
                                                                                 rstd_out, tstride, nullptr, 0);
    return cmgan_check_launch("norm_finalize_kernel");
}

// InstanceNorm tables of a ragged batch (sums from cmgan_norm_stats_varlen): group g averages over frames[g] * rows_per_frame rows
CMGAN_API int cmgan_norm_finalize_varlen(const double* sums, const int* frames, long long rows_per_frame, int T, int G, int C, const float* gamma,
                                         const float* beta, float* scale, float* shift, float* mean_out, float* rstd_out, long long tstride,
                                         void* stream) {
    CMGAN_REQUIRE(sums && frames && gamma && beta && scale && shift && rows_per_frame > 0, "cmgan_norm_finalize_varlen: bad arguments");
    norm_finalize_kernel<<<cdiv((long)G * C, 128), 128, 0, (cudaStream_t)stream>>>(sums, rows_per_frame, G, C, 0, gamma, beta, nullptr, nullptr,
                                                                                 0.f, scale, shift, mean_out, rstd_out, tstride, frames, T);
    return cmgan_check_launch("norm_finalize_kernel");
}

// S must be zeroed by the caller (G*C*2 doubles)
CMGAN_API int cmgan_norm_bwd_reduce(const float* x, long long ldx, const float* dact, long long ldd, int G, long long rows_per_group,
                                    int C, int act, const float* scale, const float* shift, const float* mean, const float* rstd,
                                    long long tstride, const float* slope, double* S, float* dslope, void* stream) {
    CMGAN_REQUIRE(x && dact && scale && shift && mean && rstd && S, "cmgan_norm_bwd_reduce: null pointer");
    act &= 15;          // bit 4 is the tf32-rounding request of cmgan_norm_bwd_apply
    CMGAN_REQUIRE(C >= 1 && C <= 256 && 256 % C == 0, "cmgan_norm_bwd_reduce: C=%d unsupported", C);
    if (G == 0 || rows_per_group == 0) return 0;
    if (C % 4 == 0 && ldx % 4 == 0 && ldd % 4 == 0 && tstride % 4 == 0 &&
        ((((uintptr_t)x) | ((uintptr_t)dact) | ((uintptr_t)scale) | ((uintptr_t)shift) | ((uintptr_t)mean) | ((uintptr_t)rstd) | ((uintptr_t)slope)) & 15) == 0) {
        const int nrg4 = 256 / (C / 4);
        const int chunk4 = nrg4 * 16;
        dim3 grid4(cdiv(rows_per_group, chunk4), G);
        norm_bwd_reduce4_kernel<<<grid4, 256, 0, (cudaStream_t)stream>>>(x, ldx, dact, ldd, rows_per_group, C, chunk4, act, scale, shift, mean, rstd,
                                                                        tstride, slope, S, dslope);
        return cmgan_check_launch("norm_bwd_reduce4_kernel");
    }
    int nrg = 256 / C;
    int chunk = nrg * 64;
    dim3 grid(cdiv(rows_per_group, chunk), G);
    norm_bwd_reduce_kernel<<<grid, 256, 256 * 3 * sizeof(double), (cudaStream_t)stream>>>(x, ldx, dact, ldd, rows_per_group, C, chunk, act,
                                                                                         scale, shift, mean, rstd, tstride, slope, S, dslope);
    return cmgan_check_launch("norm_bwd_reduce_kernel");
}

CMGAN_API int cmgan_norm_bwd_apply(const float* x, long long ldx, const float* dact, long long ldd, int G, long long rows_per_group,
                                   int C, int act, int use_batch_stats, const float* scale, const float* shift, const float* mean,
                                   const float* rstd, long long tstride, const float* slope, const double* S, float* dx,
                                   long long lddx, float* dgamma, float* dbeta, void* stream) {
    CMGAN_REQUIRE(x && dact && scale && shift && mean && rstd && S && dx, "cmgan_norm_bwd_apply: null pointer");
    const int rnd = (act >> 4) & 1;       // act | 16: dx feeds tensor-core contractions, round it to tf32 (nearest) on store
    act &= 15;
    CMGAN_REQUIRE(C >= 1 && C <= 256 && 256 % C == 0, "cmgan_norm_bwd_apply: C=%d unsupported", C);
    if (G == 0 || rows_per_group == 0) return 0;
    if (C % 4 == 0 && ldx % 4 == 0 && ldd % 4 == 0 && lddx % 4 == 0 && tstride % 4 == 0 &&
        ((((uintptr_t)x) | ((uintptr_t)dact) | ((uintptr_t)dx) | ((uintptr_t)scale) | ((uintptr_t)shift) | ((uintptr_t)mean) | ((uintptr_t)rstd) |
          ((uintptr_t)slope)) & 15) == 0) {
        const int nrg4 = 256 / (C / 4);
        const int chunk4 = nrg4 * 16;
        dim3 grid4(cdiv(rows_per_group, chunk4), G);
        norm_bwd_apply4_kernel<<<grid4, 256, 0, (cudaStream_t)stream>>>(x, ldx, dact, ldd, rows_per_group, C, chunk4, act, use_batch_stats, scale, shift,
                                                                       mean, rstd, tstride, slope, S, dx, lddx, dgamma, dbeta, rnd);
        return cmgan_check_launch("norm_bwd_apply4_kernel");
    }
    const int nrg = 256 / C;
    const int chunk = nrg * 32;
    dim3 grid(cdiv(rows_per_group, chunk), G);
    norm_bwd_apply_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(x, ldx, dact, ldd, rows_per_group, C, chunk, act, use_batch_stats, scale, shift,
                                                                 mean, rstd, tstride, slope, S, dx, lddx, dgamma, dbeta, rnd);
    return cmgan_check_launch("norm_bwd_apply_kernel");
}

CMGAN_API int cmgan_norm_apply(const float* x, long long ldx, int G, long long rows_per_group, int C, int act, const float* scale,
                               const float* shift, long long tstride, const float* slope, float* y, long long ldy, void* stream) {
    CMGAN_REQUIRE(x && y && scale && shift, "cmgan_norm_apply: null pointer");
    long total = (long)G * rows_per_group * C;
    if (total == 0) return 0;
    const bool vec = C % 4 == 0 && ldx % 4 == 0 && ldy % 4 == 0 && tstride % 4 == 0 &&
                     ((((uintptr_t)x) | ((uintptr_t)y) | ((uintptr_t)scale) | ((uintptr_t)shift) | ((uintptr_t)slope)) & 15) == 0;
    if (vec) norm_apply_kernel<4><<<cdiv(total / 4, 256), 256, 0, (cudaStream_t)stream>>>(x, ldx, rows_per_group, G, C, act, scale, shift, tstride, slope, y, ldy);
    else norm_apply_kernel<1><<<cdiv(total, 256), 256, 0, (cudaStream_t)stream>>>(x, ldx, rows_per_group, G, C, act, scale, shift, tstride, slope, y, ldy);
    return cmgan_check_launch("norm_apply_kernel");
}

CMGAN_API int cmgan_fill(float* p, long long n, float v, void* stream) {
    if (n == 0) return 0;
    fill_kernel<<<cdiv(n, 256), 256, 0, (cudaStream_t)stream>>>(p, n, v);
    return cmgan_check_launch("fill_kernel");
}

CMGAN_API int cmgan_copy_rows(const float* src, long long lds, float* dst, long long ldd, long long M, int C, void* stream) {
    CMGAN_REQUIRE(src && dst && C % 4 == 0 && lds % 4 == 0 && ldd % 4 == 0, "cmgan_copy_rows: bad arguments");
    if (M == 0) return 0;
    copy_rows_kernel<<<cdiv(M * (C / 4), 256), 256, 0, (cudaStream_t)stream>>>(src, lds, dst, ldd, M, C, 0);
    return cmgan_check_launch("copy_rows_kernel");
}

// same copy with every element rounded to tf32 (nearest) when the library is in tf32 mode: the destination is the operand of a tensor-core
// contraction (src == dst rounds in place)
CMGAN_API int cmgan_copy_rows_operand(const float* src, long long lds, float* dst, long long ldd, long long M, int C, void* stream) {
    CMGAN_REQUIRE(src && dst && C % 4 == 0 && lds % 4 == 0 && ldd % 4 == 0, "cmgan_copy_rows_operand: bad arguments");
    if (M == 0) return 0;
    if (src == dst && !g_cmgan_round_tf32) return 0;
    copy_rows_kernel<<<cdiv(M * (C / 4), 256), 256, 0, (cudaStream_t)stream>>>(src, lds, dst, ldd, M, C, g_cmgan_round_tf32);
    return cmgan_check_launch("copy_rows_kernel");
}

CMGAN_API int cmgan_add_rows(const float* src, long long lds, float* dst, long long ldd, long long M, int C, void* stream) {
    CMGAN_REQUIRE(src && dst && C % 4 == 0 && lds % 4 == 0 && ldd % 4 == 0, "cmgan_add_rows: bad arguments");
    if (M == 0) return 0;
    add_rows_kernel<<<cdiv(M * (C / 4), 256), 256, 0, (cudaStream_t)stream>>>(src, lds, dst, ldd, M, C);
    return cmgan_check_launch("add_rows_kernel");
}
