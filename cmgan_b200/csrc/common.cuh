// Shared device/host helpers for the cmgan_b200 kernels (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#define CMGAN_API extern "C" __attribute__((visibility("default")))

// ---- error channel --------------------------------------------------------------------------------
void cmgan_set_error(const char* fmt, ...);
int cmgan_check_launch(const char* what);   // cudaGetLastError() -> 0 / -1 (+ message)

#define CMGAN_REQUIRE(cond, ...)                       \
    do {                                               \
        if (!(cond)) {                                 \
            cmgan_set_error(__VA_ARGS__);              \
            return -1;                                 \
        }                                              \
    } while (0)

static inline int cdiv(long a, long b) { return (int)((a + b - 1) / b); }

// ---- tf32 operand rounding -----------------------------------------------------------------------------
// The tensor cores read fp32 operands and IGNORE the low 13 mantissa bits (truncation, a bias towards zero).  In tf32 mode every kernel
// that writes a tensor a tensor-core contraction will read therefore rounds it to nearest (cvt.rna.tf32.f32) on store.  The mode is
// library-wide (cmgan_set_tf32_rounding; cmgan_b200.ops.set_precision keeps it in step with the GEMM precision).
extern int g_cmgan_round_tf32;
__device__ __forceinline__ float cmgan_rna_tf32(float x) {
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
    return __uint_as_float(r);
}
__device__ __forceinline__ float cmgan_maybe_rna(float x, int on) { return on ? cmgan_rna_tf32(x) : x; }

// ---- math ----------------------------------------------------------------------------------------
// 1 / (1 + 2^(-x log2 e)) on the raw MUFU approximations (flush-to-zero): 2 MUFU + 2 FP instructions.  __expf / __fdividef wrap the same
// two instructions in denormal / range handling (3x the instructions) that a sigmoid does not need: exp underflow gives exactly 1,
// overflow gives 1 / inf = 0.
__device__ __forceinline__ float sigmoidf_(float x) {
    float e, s;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(x * -1.4426950408889634f));
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(s) : "f"(1.0f + e));
    return s;
}
__device__ __forceinline__ float swishf_(float x) { return x * sigmoidf_(x); }
// d/dx [x * sigmoid(x)]
__device__ __forceinline__ float dswishf_(float x) {
    float s = sigmoidf_(x);
    return s * (1.0f + x * (1.0f - s));
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// ---- dropout --------------------------------------------------------------------------------------
// Counter-based keep decision: a function of (seed, element index) only, so the backward pass (and the
// test-side mask export) regenerate exactly the mask the forward pass applied.  One 32-bit hash (lowbias32 mixer)
// serves two consecutive elements (16 bits each), so the float4 epilogues pay two hashes per four elements.
__host__ __device__ __forceinline__ uint32_t cmgan_mix32(uint32_t x) {
    x ^= x >> 16; x *= 0x7feb352dU; x ^= x >> 15; x *= 0x846ca68bU; x ^= x >> 16;
    return x;
}
// effective seed of a dropout site at graph replay `counter`: a 64-bit mix (splitmix64 finaliser) of the site seed and the device step counter,
// so that neighbouring sites / consecutive steps never share a mask function (seed + counter would alias site i at step n+1 with site i+1 at step n)
__host__ __device__ __forceinline__ uint64_t cmgan_mix_seed(uint64_t seed, uint64_t counter) {
    uint64_t z = seed ^ (counter * 0x9E3779B97F4A7C15ull);
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull; z = (z ^ (z >> 27)) * 0x94D049BB133111EBull; z ^= z >> 31;
    return z;
}
__device__ __forceinline__ uint64_t cmgan_eff_seed(uint64_t seed, const unsigned long long* __restrict__ seed_dev) {
    return seed_dev ? cmgan_mix_seed(seed, __ldg(seed_dev)) : seed;
}
__host__ __device__ __forceinline__ uint32_t cmgan_seed32(uint64_t seed) { return (uint32_t)seed ^ ((uint32_t)(seed >> 32) * 0x9E3779B9u); }
__host__ __device__ __forceinline__ uint32_t cmgan_pair_hash(uint32_t seed32, uint64_t pair) { return cmgan_mix32(((uint32_t)pair * 0x9E3779B1u) ^ seed32); }
// returns 0 (dropped) or 1/(1-p) (kept); thr = p * 2^32 (0 => dropout disabled => 1); the decision uses the top 16 bits of thr
__host__ __device__ __forceinline__ float cmgan_drop_scale(uint64_t seed, uint64_t idx, uint32_t thr, float inv_keep) {
    if (thr == 0u) return 1.0f;
    const uint32_t h = cmgan_pair_hash(cmgan_seed32(seed), idx >> 1);
    const uint32_t r = (idx & 1) ? (h >> 16) : (h & 0xFFFFu);
    return r >= (thr >> 16) ? inv_keep : 0.0f;
}
// four consecutive elements starting at idx (idx % 4 == 0): two hashes
__host__ __device__ __forceinline__ void cmgan_drop_scale4(uint64_t seed, uint64_t idx, uint32_t thr, float inv_keep, float out[4]) {
    if (thr == 0u) { out[0] = out[1] = out[2] = out[3] = 1.0f; return; }
    const uint32_t s = cmgan_seed32(seed), t = thr >> 16;
    const uint32_t h0 = cmgan_pair_hash(s, idx >> 1), h1 = cmgan_pair_hash(s, (idx >> 1) + 1);
    out[0] = (h0 & 0xFFFFu) >= t ? inv_keep : 0.0f; out[1] = (h0 >> 16) >= t ? inv_keep : 0.0f;
    out[2] = (h1 & 0xFFFFu) >= t ? inv_keep : 0.0f; out[3] = (h1 >> 16) >= t ? inv_keep : 0.0f;
}

// ---- sequence geometry -----------------------------------------------------------------------------
// Activations are channel-last rows (b, t, f) -> row index (b*T + t)*F + f.  A "sequence" is either all
// t for fixed (b, f) (time axis) or all f for fixed (b, t) (frequency axis); both are described by
//   row(s, l) = (s / n_inner) * outer_stride + (s % n_inner) * inner_stride + l * tok_stride
struct SeqGeom {
    int n_seq;          // number of sequences
    int L;              // tokens per sequence
    int n_inner;        // time: F      freq: T
    long outer_stride;  // time: T*F    freq: T*F
    long inner_stride;  // time: 1      freq: F
    long tok_stride;    // time: F      freq: 1
};
__host__ __device__ __forceinline__ long seq_base(const SeqGeom& g, int s) {
    return (long)(s / g.n_inner) * g.outer_stride + (long)(s % g.n_inner) * g.inner_stride;
}
static inline SeqGeom make_seq_geom(int B, int T, int F, int axis /*0 = time, 1 = freq*/) {
    SeqGeom g;
    if (axis == 0) { g.n_seq = B * F; g.L = T; g.n_inner = F; g.outer_stride = (long)T * F; g.inner_stride = 1; g.tok_stride = F; }
    else           { g.n_seq = B * T; g.L = F; g.n_inner = T; g.outer_stride = (long)T * F; g.inner_stride = F; g.tok_stride = 1; }
    return g;
}

// ---- ragged batches (inference) ------------------------------------------------------------------------
// A ragged batch is the (B, T, F) grid padded along time: batch item b holds frames[b] valid frames, the rows t >= frames[b] are
// padding and may hold anything (NaN included).  Kernels that combine rows along time never read a padded row.
// Frame count of item b, clamped to [0, T] so that a bad length cannot move a load outside the tensor.
__device__ __forceinline__ int varlen_frames(const int* __restrict__ frames, int b, int T) {
    const int n = __ldg(frames + b);
    return n < 0 ? 0 : (n > T ? T : n);
}
// Tokens of sequence s on a ragged grid: time axis (axis 0) -> frames[b] of its batch item; frequency axis -> all of them for a valid
// frame, none for a padded one.  (s / n_inner is the batch item on both axes.)
__device__ __forceinline__ int varlen_seq_len(const SeqGeom& g, const int* __restrict__ frames, int axis, int s) {
    const int b = s / g.n_inner;
    if (axis == 0) return varlen_frames(frames, b, g.L);
    return (s % g.n_inner) < varlen_frames(frames, b, g.n_inner) ? g.L : 0;
}
