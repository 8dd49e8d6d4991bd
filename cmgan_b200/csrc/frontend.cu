// Signal front/back end and the small HBM-bound ends of TSCNet:
//   RMS normalise + reflect pad (train.py:75-87), power-law compression / un-compression (utils.py:20-39),
//   overlap-add of the inverse STFT (train.py:106-112), the generator head (generator.py:175-179 + conv_1 :53),
//   the (1,2) output convolutions of both decoders (generator.py:126,150) and the final recombination
//   (generator.py:136-139,188-196).  The framed DFT / inverse DFT themselves are GEMMs (gemm_args.h).
#include "common.cuh"
#include "../../include/cmgan_b200.h"

namespace {

constexpr int NFFT = 400, HOP = 100, NF = 201;

// ------------------------------------------------------------------ RMS scale: c[b] = sqrt(L / sum x^2)
// lens (optional, ragged batch): row b holds lens[b] <= L samples
__global__ void rms_scale_kernel(const float* __restrict__ x, long ldx, int L, float* __restrict__ c, const int* __restrict__ lens) {
    __shared__ double sm[32];
    const float* p = x + (long)blockIdx.x * ldx;
    if (lens) L = min(__ldg(lens + blockIdx.x), L);
    double s = 0.0;
    for (int i = threadIdx.x; i < L; i += blockDim.x) { float v = __ldg(p + i); s += (double)v * v; }
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < (blockDim.x >> 5); ++w) t += sm[w];
        c[blockIdx.x] = (float)sqrt((double)L / t);
    }
}

// xp[b, i] = c[b] * x[b, reflect(i - 200)], i < L + 400; zero up to Lp
__global__ void pad_reflect_kernel(const float* __restrict__ x, long ldx, int L, const float* __restrict__ c, float* __restrict__ xp, int Lp) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    int b = blockIdx.y;
    if (i >= Lp) return;
    float v = 0.f;
    if (i < L + NFFT) {
        int j = i - NFFT / 2;
        if (j < 0) j = -j;
        if (j >= L) j = 2 * (L - 1) - j;
        v = __ldg(x + (long)b * ldx + j) * (c ? c[b] : 1.f);
    }
    xp[(long)b * Lp + i] = v;
}

// ragged batch of clips, one kernel for what evaluation.py:25-29 + train.py:77-87 do to one file: row b (lens[b] > 200 samples) is
// wrap-padded with its own head to Lw = ceil(lens[b] / 100) * 100 samples, reflect-padded by 200 on both sides and scaled by c[b]:
//   xp[b, i] = c[b] * u[reflect(i - 200)], i < Lw + 400,   u[j] = x[b, j < lens[b] ? j : j - lens[b]];   zero from Lw + 400 up to Lp
__global__ void wrap_pad_reflect_kernel(const float* __restrict__ x, long ldx, const int* __restrict__ lens, const float* __restrict__ c,
                                        float* __restrict__ xp, int Lp) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int b = blockIdx.y;
    if (i >= Lp) return;
    const int L = __ldg(lens + b);
    const int Lw = (L + HOP - 1) / HOP * HOP;
    float v = 0.f;
    if (i < Lw + NFFT) {
        int j = i - NFFT / 2;
        if (j < 0) j = -j;
        if (j >= Lw) j = 2 * (Lw - 1) - j;
        if (j >= L) j -= L;
        v = __ldg(x + (long)b * ldx + j) * c[b];
    }
    xp[(long)b * Lp + i] = v;
}

// S (B*T, 402) = [re | im]  ->  planes X[b, 0/1, t, f] = S * |S|^-0.7
__global__ void compress_kernel(const float* __restrict__ S, long total /*B*T*F*/, int T, float* __restrict__ X) {
    long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    int f = (int)(i % NF);
    long bt = i / NF;
    long b = bt / T; int t = (int)(bt % T);
    float re = __ldg(S + bt * (2 * NF) + f), im = __ldg(S + bt * (2 * NF) + NF + f);
    float m2 = re * re + im * im;
    float sc = m2 > 0.f ? powf(m2, -0.35f) : 0.f;
    long o = ((b * 2) * T + t) * NF + f;
    X[o] = re * sc;
    X[o + (long)T * NF] = im * sc;
}

// un-compression of (re, im) planes (each (B, T, F) with explicit strides) -> U (B*T, 402) = [re | im] * |.|^(7/3)
__global__ void uncompress_kernel(const float* __restrict__ re_p, const float* __restrict__ im_p, long sb, long st, long sf, long total, int T,
                                  float* __restrict__ U) {
    long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    int f = (int)(i % NF);
    long bt = i / NF;
    long b = bt / T; int t = (int)(bt % T);
    long o = b * sb + t * st + f * sf;
    float re = __ldg(re_p + o), im = __ldg(im_p + o);
    float m2 = re * re + im * im;
    float sc = m2 > 0.f ? powf(m2, 7.0f / 6.0f) : 0.f;
    U[bt * (2 * NF) + f] = re * sc;
    U[bt * (2 * NF) + NF + f] = im * sc;
}

// gradient of the un-compression: dU (B*T, 402) -> d_re, d_im planes (B, T, F) contiguous
__global__ void uncompress_bwd_kernel(const float* __restrict__ re_p, const float* __restrict__ im_p, long sb, long st, long sf, long total, int T,
                                      const float* __restrict__ dU, float* __restrict__ dre, float* __restrict__ dim_, int accumulate) {
    long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    int f = (int)(i % NF);
    long bt = i / NF;
    long b = bt / T; int t = (int)(bt % T);
    long o = b * sb + t * st + f * sf;
    float re = __ldg(re_p + o), im = __ldg(im_p + o);
    float gr = __ldg(dU + bt * (2 * NF) + f), gi = __ldg(dU + bt * (2 * NF) + NF + f);
    float m2 = re * re + im * im;
    float dr = 0.f, di = 0.f;
    if (m2 > 0.f) {
        const float p = 7.0f / 3.0f;
        float mp = powf(m2, 0.5f * p);            // m^p
        float mp2 = p * mp / m2;                  // p m^(p-2)
        dr = gr * (mp + mp2 * re * re) + gi * (mp2 * re * im);
        di = gr * (mp2 * re * im) + gi * (mp + mp2 * im * im);
    }
    if (accumulate) { dre[i] += dr; dim_[i] += di; }
    else { dre[i] = dr; dim_[i] = di; }
}

// generic strided power law  Y = X * |X|^p  over a (d0, d1, d2) index space (power_compress p = -0.7, power_uncompress p = 7/3)
__global__ void power_law_kernel(const float* __restrict__ re, const float* __restrict__ im, long i0, long i1, long i2, float* __restrict__ ore,
                                 float* __restrict__ oim, long o0, long o1, long o2, int d1, int d2, long n, float half_p) {
    long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int c = (int)(i % d2); long t = i / d2; int b = (int)(t % d1); long a = t / d1;
    long io = a * i0 + b * i1 + c * i2, oo = a * o0 + b * o1 + c * o2;
    float r = __ldg(re + io), m = __ldg(im + io);
    float m2 = r * r + m * m;
    float sc = m2 > 0.f ? powf(m2, half_p) : 0.f;
    ore[oo] = r * sc; oim[oo] = m * sc;
}
// gradient: (gre, gim) at the output strides -> (dre, dim) at the input strides
__global__ void power_law_bwd_kernel(const float* __restrict__ re, const float* __restrict__ im, long i0, long i1, long i2,
                                     const float* __restrict__ gre, const float* __restrict__ gim, long o0, long o1, long o2,
                                     float* __restrict__ dre, float* __restrict__ dim_, long q0, long q1, long q2, int d1, int d2, long n, float p) {
    long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int c = (int)(i % d2); long t = i / d2; int b = (int)(t % d1); long a = t / d1;
    long io = a * i0 + b * i1 + c * i2, oo = a * o0 + b * o1 + c * o2, qo = a * q0 + b * q1 + c * q2;
    float r = __ldg(re + io), m = __ldg(im + io), gr = __ldg(gre + oo), gi = __ldg(gim + oo);
    float m2 = r * r + m * m;
    float dr = 0.f, di = 0.f;
    if (m2 > 0.f) {
        float mp = powf(m2, 0.5f * p), mp2 = p * mp / m2;
        dr = gr * (mp + mp2 * r * r) + gi * (mp2 * r * m);
        di = gr * (mp2 * r * m) + gi * (mp + mp2 * m * m);
    }
    dre[qo] = dr; dim_[qo] = di;
}

// overlap-add: y[b, n] = (sum_t frames[b, t, n + 200 - 100 t]) / env[n],  n < 100 (T - 1)
__global__ void ola_kernel(const float* __restrict__ frames, int T, const float* __restrict__ inv_env, const float* __restrict__ c_div,
                           float* __restrict__ y, long ldy) {
    int n = blockIdx.x * blockDim.x + threadIdx.x;
    int b = blockIdx.y;
    int Lout = HOP * (T - 1);
    if (n >= Lout) return;
    int p = n + NFFT / 2;                         // position in the un-trimmed signal
    int t_hi = p / HOP; if (t_hi > T - 1) t_hi = T - 1;
    int t_lo = (p - NFFT + HOP) / HOP; if (p - NFFT + 1 <= 0) t_lo = 0;
    float s = 0.f;
    for (int t = t_lo; t <= t_hi; ++t) {
        int k = p - t * HOP;
        if (k >= 0 && k < NFFT) s += __ldg(frames + ((long)b * T + t) * NFFT + k);
    }
    s *= inv_env[n];
    if (c_div) s /= c_div[b];
    y[(long)b * ldy + n] = s;
}

// overlap-add of a ragged batch: utterance b has nframes[b] <= T frames.  The window-square envelope of each utterance is summed here in
// float64, frame by frame in increasing t exactly like signal._inv_envelope (win_sq = the float64 squared window), so every sample
// equals that of the per-utterance ola_kernel.  Samples from 100 (nframes[b] - 1) on are zero.
__global__ void ola_varlen_kernel(const float* __restrict__ frames, int T, const int* __restrict__ nframes, const double* __restrict__ win_sq,
                                  const float* __restrict__ c_div, float* __restrict__ y, long ldy) {
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    const int b = blockIdx.y;
    if (n >= HOP * (T - 1)) return;
    const int Tb = min(__ldg(nframes + b), T);
    float s = 0.f;
    if (n < HOP * (Tb - 1)) {
        const int p = n + NFFT / 2;
        int t_hi = p / HOP; if (t_hi > Tb - 1) t_hi = Tb - 1;
        int t_lo = (p - NFFT + HOP) / HOP; if (p - NFFT + 1 <= 0) t_lo = 0;
        double env = 0.0;
        for (int t = t_lo; t <= t_hi; ++t) {
            int k = p - t * HOP;
            if (k >= 0 && k < NFFT) {
                s += __ldg(frames + ((long)b * T + t) * NFFT + k);
                env += __ldg(win_sq + k);
            }
        }
        s *= (float)(1.0 / env);
        if (c_div) s /= c_div[b];
    }
    y[(long)b * ldy + n] = s;
}

// gradient of overlap-add: dframes[b, t, k] = dy[b, 100 t + k - 200] / env (zero outside the trimmed range)
__global__ void ola_bwd_kernel(const float* __restrict__ dy, long lddy, int T, const float* __restrict__ inv_env, float* __restrict__ dframes) {
    long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    int b = blockIdx.y;
    if (i >= (long)T * NFFT) return;
    int t = (int)(i / NFFT), k = (int)(i % NFFT);
    int n = t * HOP + k - NFFT / 2;
    float v = 0.f;
    if (n >= 0 && n < HOP * (T - 1)) v = __ldg(dy + (long)b * lddy + n) * inv_env[n];
    dframes[(long)b * T * NFFT + i] = v;
}

// ------------------------------------------------------------------ generator head: mag + 1x1 conv 3 -> 64 (raw, pre-norm)
// x (B, 2, T, F) with strides; out rows (b, t, f) with leading dimension ldo
__global__ void head_conv_kernel(const float* __restrict__ x, long sb, long sc, long st, long sf, int T, int F, long M,
                                 const float* __restrict__ w /*(64,3)*/, const float* __restrict__ bias, float* __restrict__ out, long ldo) {
    long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
    long m = idx >> 4; int c4 = (int)(idx & 15) * 4;
    if (m >= M) return;
    int f = (int)(m % F); long bt = m / F; int t = (int)(bt % T); long b = bt / T;
    long o = b * sb + t * st + f * sf;
    float re = __ldg(x + o), im = __ldg(x + o + sc);
    float mag = sqrtf(re * re + im * im);
    float r[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        int n = c4 + j;
        r[j] = fmaf(__ldg(w + n * 3), mag, fmaf(__ldg(w + n * 3 + 1), re, fmaf(__ldg(w + n * 3 + 2), im, __ldg(bias + n))));
    }
    *reinterpret_cast<float4*>(out + m * ldo + c4) = make_float4(r[0], r[1], r[2], r[3]);
}

// dW (64,3) += sum_m draw[m, n] * in_j[m];  dbias[n] += sum_m draw[m, n]
__global__ void head_conv_wgrad_kernel(const float* __restrict__ x, long sb, long sc, long st, long sf, int T, int F, long M,
                                       const float* __restrict__ draw, long ldd, int rows_per_block, float* __restrict__ dw, float* __restrict__ db) {
    __shared__ float sm[4][4][64];
    int n = threadIdx.x & 63, rg = threadIdx.x >> 6;       // 256 threads: 4 row groups x 64 channels
    long m_beg = (long)blockIdx.x * rows_per_block, m_end = m_beg + rows_per_block < M ? m_beg + rows_per_block : M;
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
    for (long m = m_beg + rg; m < m_end; m += 4) {
        int f = (int)(m % F); long bt = m / F; int t = (int)(bt % T); long b = bt / T;
        long o = b * sb + t * st + f * sf;
        float re = __ldg(x + o), im = __ldg(x + o + sc);
        float mag = sqrtf(re * re + im * im);
        float d = __ldg(draw + m * ldd + n);
        a0 = fmaf(d, mag, a0); a1 = fmaf(d, re, a1); a2 = fmaf(d, im, a2); a3 += d;
    }
    sm[rg][0][n] = a0; sm[rg][1][n] = a1; sm[rg][2][n] = a2; sm[rg][3][n] = a3;
    __syncthreads();
    if (rg == 0) {
        float s0 = 0, s1 = 0, s2 = 0, s3 = 0;
        for (int g = 0; g < 4; ++g) { s0 += sm[g][0][n]; s1 += sm[g][1][n]; s2 += sm[g][2][n]; s3 += sm[g][3][n]; }
        atomicAdd(dw + n * 3, s0); atomicAdd(dw + n * 3 + 1, s1); atomicAdd(dw + n * 3 + 2, s2); atomicAdd(db + n, s3);
    }
}

// ------------------------------------------------------------------ (1,2) output convolutions, 64 -> NOUT (1 or 2)
// in rows (b, t, f'), f' < Fin = Fout + 1, 64 channels, optional InstanceNorm+PReLU prologue (scale/shift per (b, c)).
// out[(b,t,f), j] = bias[j] + sum_{dj<2} sum_c act(in[(b,t,f+dj), c]) * w[j, c, 0, dj].  One warp per output pixel.
template <int NOUT>
__global__ void rowdot_fwd_kernel(const float* __restrict__ in, int T, int Fout, long npix, const float* __restrict__ scale,
                                  const float* __restrict__ shift, const float* __restrict__ slope, const float* __restrict__ w,
                                  const float* __restrict__ bias, float* __restrict__ out) {
    long pix = (long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    int lane = threadIdx.x & 31;
    if (pix >= npix) return;
    int f = (int)(pix % Fout); long bt = pix / Fout; long b = bt / T;
    const int Fin = Fout + 1;
    int k = lane * 4, dj = k >> 6, c = k & 63;
    float4 v = __ldg(reinterpret_cast<const float4*>(in + (bt * Fin + f) * 64) + lane);
    float a[4] = {v.x, v.y, v.z, v.w};
    if (scale) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            float z = a[i] * __ldg(scale + b * 64 + c + i) + __ldg(shift + b * 64 + c + i);
            a[i] = z >= 0.f ? z : z * __ldg(slope + c + i);
        }
    }
#pragma unroll
    for (int j = 0; j < NOUT; ++j) {
        float s = 0.f;
#pragma unroll
        for (int i = 0; i < 4; ++i) s = fmaf(a[i], __ldg(w + (j * 64 + c + i) * 2 + dj), s);
        s = warp_sum(s);
        if (lane == 0) out[pix * NOUT + j] = s + __ldg(bias + j);
    }
}

// backward of the above.  dact (B,T,Fin,64) = grad wrt act(in) (overwritten); dw (NOUT,64,1,2), dbias accumulated.
// One warp per input row (b, t, f'); lane owns channels 2*lane, 2*lane+1.
template <int NOUT>
__global__ void rowdot_bwd_kernel(const float* __restrict__ in, int T, int Fout, long nrows, const float* __restrict__ scale,
                                  const float* __restrict__ shift, const float* __restrict__ slope, const float* __restrict__ w,
                                  const float* __restrict__ dout, int rows_per_warp, float* __restrict__ dact, float* __restrict__ dw,
                                  float* __restrict__ dbias) {
    __shared__ float sm[8][NOUT * 2 * 64];
    int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    const int Fin = Fout + 1;
    float wr[NOUT][2][2];     // [j][dj][ch]
    float acc[NOUT][2][2];
    float bacc[NOUT];
#pragma unroll
    for (int j = 0; j < NOUT; ++j) {
        bacc[j] = 0.f;
#pragma unroll
        for (int dj = 0; dj < 2; ++dj)
#pragma unroll
            for (int e = 0; e < 2; ++e) { wr[j][dj][e] = __ldg(w + (j * 64 + 2 * lane + e) * 2 + dj); acc[j][dj][e] = 0.f; }
    }
    long r0 = ((long)blockIdx.x * nw + warp) * rows_per_warp;
    for (int it = 0; it < rows_per_warp; ++it) {
        long row = r0 + it;
        if (row >= nrows) break;
        int fp = (int)(row % Fin); long bt = row / Fin; long b = bt / T;
        float2 v = __ldg(reinterpret_cast<const float2*>(in + row * 64) + lane);
        float a[2] = {v.x, v.y};
        if (scale) {
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                int c = 2 * lane + e;
                float z = a[e] * __ldg(scale + b * 64 + c) + __ldg(shift + b * 64 + c);
                a[e] = z >= 0.f ? z : z * __ldg(slope + c);
            }
        }
        float g[2] = {0.f, 0.f};
#pragma unroll
        for (int j = 0; j < NOUT; ++j) {
            float d0 = fp < Fout ? __ldg(dout + (bt * Fout + fp) * NOUT + j) : 0.f;      // this row is tap dj = 0 of pixel fp
            float d1 = fp >= 1 ? __ldg(dout + (bt * Fout + fp - 1) * NOUT + j) : 0.f;    // and tap dj = 1 of pixel fp - 1
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                g[e] = fmaf(d0, wr[j][0][e], fmaf(d1, wr[j][1][e], g[e]));
                acc[j][0][e] = fmaf(d0, a[e], acc[j][0][e]);
                acc[j][1][e] = fmaf(d1, a[e], acc[j][1][e]);
            }
            if (lane == 0) bacc[j] += d0;
        }
        reinterpret_cast<float2*>(dact + row * 64)[lane] = make_float2(g[0], g[1]);
    }
#pragma unroll
    for (int j = 0; j < NOUT; ++j)
#pragma unroll
        for (int dj = 0; dj < 2; ++dj)
#pragma unroll
            for (int e = 0; e < 2; ++e) sm[warp][(j * 2 + dj) * 64 + 2 * lane + e] = acc[j][dj][e];
    __syncthreads();
    for (int i = threadIdx.x; i < NOUT * 2 * 64; i += blockDim.x) {
        float s = 0.f;
        for (int wv = 0; wv < nw; ++wv) s += sm[wv][i];
        int j = i / 128, dj = (i / 64) & 1, c = i & 63;
        atomicAdd(dw + (j * 64 + c) * 2 + dj, s);
    }
    if (lane == 0) {
#pragma unroll
        for (int j = 0; j < NOUT; ++j) atomicAdd(dbias + j, bacc[j]);
    }
}

// ------------------------------------------------------------------ recombination (mask tail + complex add)
// m1 (B*T*F) raw (1,2)-conv output of the mask branch; IN(1) scale/shift per b; PReLU(1) a1; 1x1 conv (fcw, fcb);
// PReLU with one slope per frequency; final = mask * x + cplx.
struct MaskTail { const float* scale; const float* shift; const float* a1; const float* fcw; const float* fcb; const float* slope_f; };

__global__ void recombine_kernel(const float* __restrict__ m1, MaskTail mt, const float* __restrict__ x, long sb, long sc, long st, long sf,
                                 const float* __restrict__ cplx, int T, int F, long M, float* __restrict__ fr, float* __restrict__ fi) {
    long m = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= M) return;
    int f = (int)(m % F); long bt = m / F; int t = (int)(bt % T); long b = bt / T;
    float z = __ldg(m1 + m) * mt.scale[b] + mt.shift[b];
    if (z < 0.f) z *= mt.a1[0];
    float z2 = fmaf(mt.fcw[0], z, mt.fcb[0]);
    float mask = z2 >= 0.f ? z2 : z2 * __ldg(mt.slope_f + f);
    long o = b * sb + t * st + f * sf;
    float re = __ldg(x + o), im = __ldg(x + o + sc);
    float2 c = __ldg(reinterpret_cast<const float2*>(cplx) + m);
    fr[m] = fmaf(mask, re, c.x);
    fi[m] = fmaf(mask, im, c.y);
}

// backward: dfr, dfi with strides (gb, gt, gf) -> dcplx (M, 2), dz (M) = grad wrt the IN(1)+PReLU(1) output;
// dslope_f (F), dfcw, dfcb accumulated
__global__ void recombine_bwd_kernel(const float* __restrict__ m1, MaskTail mt, const float* __restrict__ x, long sb, long sc, long st, long sf,
                                     const float* __restrict__ dfr, const float* __restrict__ dfi, long gb, long gt, long gf, int T, int F,
                                     long M, float* __restrict__ dcplx, float* __restrict__ dz, float* __restrict__ dslope_f,
                                     float* __restrict__ dfcw, float* __restrict__ dfcb) {
    long m = (long)blockIdx.x * blockDim.x + threadIdx.x;
    float pw = 0.f, pb = 0.f;
    if (m < M) {
        int f = (int)(m % F); long bt = m / F; int t = (int)(bt % T); long b = bt / T;
        float z = __ldg(m1 + m) * mt.scale[b] + mt.shift[b];
        if (z < 0.f) z *= mt.a1[0];
        float z2 = fmaf(mt.fcw[0], z, mt.fcb[0]);
        long o = b * sb + t * st + f * sf;
        float re = __ldg(x + o), im = __ldg(x + o + sc);
        long go = b * gb + t * gt + f * gf;
        float gr = __ldg(dfr + go), gi = __ldg(dfi + go);
        reinterpret_cast<float2*>(dcplx)[m] = make_float2(gr, gi);
        float dmask = gr * re + gi * im;
        float dz2 = dmask;
        if (z2 < 0.f) { dz2 = dmask * __ldg(mt.slope_f + f); atomicAdd(dslope_f + f, dmask * z2); }
        pw = dz2 * z; pb = dz2;
        dz[m] = dz2 * mt.fcw[0];
    }
    pw = warp_sum(pw); pb = warp_sum(pb);
    if ((threadIdx.x & 31) == 0) { atomicAdd(dfcw, pw); atomicAdd(dfcb, pb); }
}

}  // namespace

// ------------------------------------------------------------------ C ABI
CMGAN_API int cmgan_rms_scale(const float* x, long long ldx, int B, int L, float* c, void* stream) {
    CMGAN_REQUIRE(x && c && L > 0, "cmgan_rms_scale: bad arguments");
    if (B == 0) return 0;
    rms_scale_kernel<<<B, 256, 0, (cudaStream_t)stream>>>(x, ldx, L, c, nullptr);
    return cmgan_check_launch("rms_scale_kernel");
}

// ragged batch: c[b] = sqrt(lens[b] / sum of the first lens[b] samples of row b squared); ldx >= every lens[b]
CMGAN_API int cmgan_rms_scale_varlen(const float* x, long long ldx, int B, const int* lens, float* c, void* stream) {
    CMGAN_REQUIRE(x && lens && c && ldx > 0, "cmgan_rms_scale_varlen: bad arguments");
    if (B == 0) return 0;
    rms_scale_kernel<<<B, 256, 0, (cudaStream_t)stream>>>(x, ldx, (int)ldx, c, lens);
    return cmgan_check_launch("rms_scale_kernel");
}

// ragged batch: xp (B, Lp) = wrap pad to a multiple of 100 + reflect pad 200 + scale by c[b] (wrap_pad_reflect_kernel);
// needs 200 < lens[b] and Lp >= ceil(lens[b] / 100) * 100 + 400 for every b
CMGAN_API int cmgan_wrap_pad_reflect_varlen(const float* x, long long ldx, int B, const int* lens, const float* c, float* xp, int Lp, void* stream) {
    CMGAN_REQUIRE(x && lens && c && xp && Lp > 0, "cmgan_wrap_pad_reflect_varlen: bad arguments");
    if (B == 0) return 0;
    dim3 grid(cdiv(Lp, 256), B);
    wrap_pad_reflect_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(x, ldx, lens, c, xp, Lp);
    return cmgan_check_launch("wrap_pad_reflect_kernel");
}

// xp (B, Lp): reflect-padded (200 each side) and scaled by c[b] (c may be null); Lp >= L + 400, zero filled beyond
CMGAN_API int cmgan_pad_reflect(const float* x, long long ldx, int B, int L, const float* c, float* xp, int Lp, void* stream) {
    CMGAN_REQUIRE(x && xp && L > 200 && Lp >= L + 400, "cmgan_pad_reflect: need L > 200 and Lp >= L + 400 (L=%d Lp=%d)", L, Lp);
    if (B == 0) return 0;
    dim3 grid(cdiv(Lp, 256), B);
    pad_reflect_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(x, ldx, L, c, xp, Lp);
    return cmgan_check_launch("pad_reflect_kernel");
}

CMGAN_API int cmgan_compress(const float* S, int B, int T, float* X, void* stream) {
    CMGAN_REQUIRE(S && X, "cmgan_compress: null pointer");
    long total = (long)B * T * NF;
    if (total == 0) return 0;
    compress_kernel<<<cdiv(total, 256), 256, 0, (cudaStream_t)stream>>>(S, total, T, X);
    return cmgan_check_launch("compress_kernel");
}

CMGAN_API int cmgan_uncompress(const float* re, const float* im, long long sb, long long st, long long sf, int B, int T, float* U, void* stream) {
    CMGAN_REQUIRE(re && im && U, "cmgan_uncompress: null pointer");
    long total = (long)B * T * NF;
    if (total == 0) return 0;
    uncompress_kernel<<<cdiv(total, 256), 256, 0, (cudaStream_t)stream>>>(re, im, sb, st, sf, total, T, U);
    return cmgan_check_launch("uncompress_kernel");
}

CMGAN_API int cmgan_uncompress_bwd(const float* re, const float* im, long long sb, long long st, long long sf, int B, int T, const float* dU,
                                   float* dre, float* dim_, int accumulate, void* stream) {
    CMGAN_REQUIRE(re && im && dU && dre && dim_, "cmgan_uncompress_bwd: null pointer");
    long total = (long)B * T * NF;
    if (total == 0) return 0;
    uncompress_bwd_kernel<<<cdiv(total, 256), 256, 0, (cudaStream_t)stream>>>(re, im, sb, st, sf, total, T, dU, dre, dim_, accumulate);
    return cmgan_check_launch("uncompress_bwd_kernel");
}

CMGAN_API int cmgan_ola(const float* frames, int B, int T, const float* inv_env, const float* c_div, float* y, long long ldy, void* stream) {
    CMGAN_REQUIRE(frames && inv_env && y && T >= 2, "cmgan_ola: bad arguments");
    if (B == 0) return 0;
    dim3 grid(cdiv((long)HOP * (T - 1), 256), B);
    ola_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(frames, T, inv_env, c_div, y, ldy);
    return cmgan_check_launch("ola_kernel");
}

// ragged batch: frames (B*T, 400), utterance b has nframes[b] frames (2 <= nframes[b] <= T); win_sq = 400 doubles (squared Hamming window)
CMGAN_API int cmgan_ola_varlen(const float* frames, int B, int T, const int* nframes, const double* win_sq, const float* c_div, float* y,
                               long long ldy, void* stream) {
    CMGAN_REQUIRE(frames && nframes && win_sq && y && T >= 2, "cmgan_ola_varlen: bad arguments");
    if (B == 0) return 0;
    dim3 grid(cdiv((long)HOP * (T - 1), 256), B);
    ola_varlen_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(frames, T, nframes, win_sq, c_div, y, ldy);
    return cmgan_check_launch("ola_varlen_kernel");
}

CMGAN_API int cmgan_ola_bwd(const float* dy, long long lddy, int B, int T, const float* inv_env, float* dframes, void* stream) {
    CMGAN_REQUIRE(dy && inv_env && dframes && T >= 2, "cmgan_ola_bwd: bad arguments");
    if (B == 0) return 0;
    dim3 grid(cdiv((long)T * NFFT, 256), B);
    ola_bwd_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(dy, lddy, T, inv_env, dframes);
    return cmgan_check_launch("ola_bwd_kernel");
}

CMGAN_API int cmgan_head_conv(const float* x, long long sb, long long sc, long long st, long long sf, int B, int T, int F, const float* w,
                              const float* bias, float* out, long long ldo, void* stream) {
    CMGAN_REQUIRE(x && w && bias && out && ldo % 4 == 0, "cmgan_head_conv: bad arguments");
    long M = (long)B * T * F;
    if (M == 0) return 0;
    head_conv_kernel<<<cdiv(M * 16, 256), 256, 0, (cudaStream_t)stream>>>(x, sb, sc, st, sf, T, F, M, w, bias, out, ldo);
    return cmgan_check_launch("head_conv_kernel");
}

CMGAN_API int cmgan_head_conv_wgrad(const float* x, long long sb, long long sc, long long st, long long sf, int B, int T, int F,
                                    const float* draw, long long ldd, float* dw, float* db, void* stream) {
    CMGAN_REQUIRE(x && draw && dw && db, "cmgan_head_conv_wgrad: null pointer");
    long M = (long)B * T * F;
    if (M == 0) return 0;
    const int rpb = 512;
    head_conv_wgrad_kernel<<<cdiv(M, rpb), 256, 0, (cudaStream_t)stream>>>(x, sb, sc, st, sf, T, F, M, draw, ldd, rpb, dw, db);
    return cmgan_check_launch("head_conv_wgrad_kernel");
}

CMGAN_API int cmgan_rowdot_fwd(const float* in, int B, int T, int Fout, int nout, const float* scale, const float* shift, const float* slope,
                               const float* w, const float* bias, float* out, void* stream) {
    CMGAN_REQUIRE(in && w && bias && out && (nout == 1 || nout == 2), "cmgan_rowdot_fwd: bad arguments");
    long npix = (long)B * T * Fout;
    if (npix == 0) return 0;
    if (nout == 1) rowdot_fwd_kernel<1><<<cdiv(npix, 8), 256, 0, (cudaStream_t)stream>>>(in, T, Fout, npix, scale, shift, slope, w, bias, out);
    else rowdot_fwd_kernel<2><<<cdiv(npix, 8), 256, 0, (cudaStream_t)stream>>>(in, T, Fout, npix, scale, shift, slope, w, bias, out);
    return cmgan_check_launch("rowdot_fwd_kernel");
}

CMGAN_API int cmgan_rowdot_bwd(const float* in, int B, int T, int Fout, int nout, const float* scale, const float* shift, const float* slope,
                               const float* w, const float* dout, float* dact, float* dw, float* dbias, void* stream) {
    CMGAN_REQUIRE(in && w && dout && dact && dw && dbias && (nout == 1 || nout == 2), "cmgan_rowdot_bwd: bad arguments");
    long nrows = (long)B * T * (Fout + 1);
    if (nrows == 0) return 0;
    const int rpw = 32;
    if (nout == 1) rowdot_bwd_kernel<1><<<cdiv(nrows, 8 * rpw), 256, 0, (cudaStream_t)stream>>>(in, T, Fout, nrows, scale, shift, slope, w, dout, rpw, dact, dw, dbias);
    else rowdot_bwd_kernel<2><<<cdiv(nrows, 8 * rpw), 256, 0, (cudaStream_t)stream>>>(in, T, Fout, nrows, scale, shift, slope, w, dout, rpw, dact, dw, dbias);
    return cmgan_check_launch("rowdot_bwd_kernel");
}

CMGAN_API int cmgan_recombine(const float* m1, const float* in_scale, const float* in_shift, const float* a1, const float* fcw, const float* fcb,
                              const float* slope_f, const float* x, long long sb, long long sc, long long st, long long sf, const float* cplx,
                              int B, int T, int F, float* fr, float* fi, void* stream) {
    CMGAN_REQUIRE(m1 && in_scale && in_shift && a1 && fcw && fcb && slope_f && x && cplx && fr && fi, "cmgan_recombine: null pointer");
    long M = (long)B * T * F;
    if (M == 0) return 0;
    MaskTail mt{in_scale, in_shift, a1, fcw, fcb, slope_f};
    recombine_kernel<<<cdiv(M, 256), 256, 0, (cudaStream_t)stream>>>(m1, mt, x, sb, sc, st, sf, cplx, T, F, M, fr, fi);
    return cmgan_check_launch("recombine_kernel");
}

CMGAN_API int cmgan_recombine_bwd(const float* m1, const float* in_scale, const float* in_shift, const float* a1, const float* fcw,
                                  const float* fcb, const float* slope_f, const float* x, long long sb, long long sc, long long st, long long sf,
                                  const float* dfr, const float* dfi, long long gb, long long gt, long long gf, int B, int T, int F,
                                  float* dcplx, float* dz, float* dslope_f, float* dfcw, float* dfcb, void* stream) {
    CMGAN_REQUIRE(m1 && in_scale && in_shift && a1 && fcw && fcb && slope_f && x && dfr && dfi && dcplx && dz && dslope_f && dfcw && dfcb,
                  "cmgan_recombine_bwd: null pointer");
    long M = (long)B * T * F;
    if (M == 0) return 0;
    MaskTail mt{in_scale, in_shift, a1, fcw, fcb, slope_f};
    recombine_bwd_kernel<<<cdiv(M, 256), 256, 0, (cudaStream_t)stream>>>(m1, mt, x, sb, sc, st, sf, dfr, dfi, gb, gt, gf, T, F, M, dcplx, dz,
                                                                        dslope_f, dfcw, dfcb);
    return cmgan_check_launch("recombine_bwd_kernel");
}

// Y = X |X|^p with explicit element strides (utils.power_compress / power_uncompress as free functions)
CMGAN_API int cmgan_power_law(const float* re, const float* im, long long i0, long long i1, long long i2, float* ore, float* oim, long long o0,
                              long long o1, long long o2, int d0, int d1, int d2, float p, void* stream) {
    CMGAN_REQUIRE(re && im && ore && oim, "cmgan_power_law: null pointer");
    long n = (long)d0 * d1 * d2;
    if (n == 0) return 0;
    power_law_kernel<<<cdiv(n, 256), 256, 0, (cudaStream_t)stream>>>(re, im, i0, i1, i2, ore, oim, o0, o1, o2, d1, d2, n, 0.5f * p);
    return cmgan_check_launch("power_law_kernel");
}

CMGAN_API int cmgan_power_law_bwd(const float* re, const float* im, long long i0, long long i1, long long i2, const float* gre, const float* gim,
                                  long long o0, long long o1, long long o2, float* dre, float* dim_, long long q0, long long q1, long long q2,
                                  int d0, int d1, int d2, float p, void* stream) {
    CMGAN_REQUIRE(re && im && gre && gim && dre && dim_, "cmgan_power_law_bwd: null pointer");
    long n = (long)d0 * d1 * d2;
    if (n == 0) return 0;
    power_law_bwd_kernel<<<cdiv(n, 256), 256, 0, (cudaStream_t)stream>>>(re, im, i0, i1, i2, gre, gim, o0, o1, o2, dre, dim_, q0, q1, q2, d1, d2, n, p);
    return cmgan_check_launch("power_law_bwd_kernel");
}
