// Module-level entry point: TSCNet.forward in inference mode (eval: BatchNorm running statistics, no dropout) as ONE C call over the
// kernels of this library -- the boundary SURVEY 8(b) asks for a non-Python host: raw device pointers, explicit strides, a caller-owned
// workspace sized by a query, int status + cmgan_last_error(), everything enqueued on the caller's stream, no allocation, no sync.
// Reference: generator.py:160-196 (TSCNet), :50-69 (DenseEncoder), :6-47 (DilatedDenseNet), :72-99 (TSCB), :122-156 (decoders),
// conformer.py:182-222 (ConformerBlock).  The launch sequence is the one cmgan_b200/network.py + conformer_block.py issue from Python
// (same kernels, same order), so the results are bit-identical to the nn.Module path.
//
// Parameters: one flat fp32 block holding every floating-point tensor of the reference's state_dict, in state_dict order, each tensor
// starting at a multiple of 4 floats (cmgan_tscnet_param_info enumerates key / offset / element count; the int64 num_batches_tracked
// buffers are not part of it).
#include <cstring>
#include <string>
#include <unordered_map>
#include <vector>

#include "common.cuh"
#include "../../include/cmgan_b200.h"

namespace {

constexpr int C = 64, CAT = 320, NFEAT = 201;

struct Entry { std::string key; long long off, numel; };

struct Table {
    std::vector<Entry> e;
    long long total = 0;
    void add(const std::string& k, long long n) {
        e.push_back({k, total, n});
        total += (n + 3) / 4 * 4;
    }
    void norm_prelu(const std::string& p, const char* norm, const char* prelu) {
        add(p + norm + ".weight", C); add(p + norm + ".bias", C); add(p + prelu + ".weight", C);
    }
    void dense_block(const std::string& p) {            // generator.py:6-37
        for (int i = 1; i <= 4; ++i) {
            const std::string s = std::to_string(i);
            add(p + "conv" + s + ".weight", (long long)C * C * i * 6); add(p + "conv" + s + ".bias", C);
            add(p + "norm" + s + ".weight", C); add(p + "norm" + s + ".bias", C); add(p + "prelu" + s + ".weight", C);
        }
    }
    void feed_forward(const std::string& p) {           // conformer.py:136-148 wrapped by Scale(PreNorm(...)) :54-72
        add(p + "fn.fn.net.0.weight", 4 * C * C); add(p + "fn.fn.net.0.bias", 4 * C);
        add(p + "fn.fn.net.3.weight", 4 * C * C); add(p + "fn.fn.net.3.bias", C);
        add(p + "fn.norm.weight", C); add(p + "fn.norm.bias", C);
    }
    void conformer(const std::string& p) {              // conformer.py:182-214
        feed_forward(p + "ff1.");
        add(p + "attn.fn.to_q.weight", C * C); add(p + "attn.fn.to_kv.weight", 2 * C * C);
        add(p + "attn.fn.to_out.weight", C * C); add(p + "attn.fn.to_out.bias", C);
        add(p + "attn.fn.rel_pos_emb.weight", 1025 * 16);
        add(p + "attn.norm.weight", C); add(p + "attn.norm.bias", C);
        add(p + "conv.net.0.weight", C); add(p + "conv.net.0.bias", C);
        add(p + "conv.net.2.weight", 4 * C * C); add(p + "conv.net.2.bias", 4 * C);
        add(p + "conv.net.4.conv.weight", 2 * C * 31); add(p + "conv.net.4.conv.bias", 2 * C);
        add(p + "conv.net.5.weight", 2 * C); add(p + "conv.net.5.bias", 2 * C);
        add(p + "conv.net.5.running_mean", 2 * C); add(p + "conv.net.5.running_var", 2 * C);
        add(p + "conv.net.7.weight", 2 * C * C); add(p + "conv.net.7.bias", C);
        feed_forward(p + "ff2.");
        add(p + "post_norm.weight", C); add(p + "post_norm.bias", C);
    }
    Table() {
        add("dense_encoder.conv_1.0.weight", C * 3); add("dense_encoder.conv_1.0.bias", C);
        norm_prelu("dense_encoder.conv_1.", "1", "2");
        dense_block("dense_encoder.dilated_dense.");
        add("dense_encoder.conv_2.0.weight", C * C * 3); add("dense_encoder.conv_2.0.bias", C);
        norm_prelu("dense_encoder.conv_2.", "1", "2");
        for (int i = 1; i <= 4; ++i) {
            conformer("TSCB_" + std::to_string(i) + ".time_conformer.");
            conformer("TSCB_" + std::to_string(i) + ".freq_conformer.");
        }
        dense_block("mask_decoder.dense_block.");
        add("mask_decoder.sub_pixel.conv.weight", 2 * C * C * 3); add("mask_decoder.sub_pixel.conv.bias", 2 * C);
        add("mask_decoder.conv_1.weight", C * 2); add("mask_decoder.conv_1.bias", 1);
        add("mask_decoder.norm.weight", 1); add("mask_decoder.norm.bias", 1);
        add("mask_decoder.prelu.weight", 1);
        add("mask_decoder.final_conv.weight", 1); add("mask_decoder.final_conv.bias", 1);
        add("mask_decoder.prelu_out.weight", NFEAT);
        dense_block("complex_decoder.dense_block.");
        add("complex_decoder.sub_pixel.conv.weight", 2 * C * C * 3); add("complex_decoder.sub_pixel.conv.bias", 2 * C);
        add("complex_decoder.prelu.weight", C);
        add("complex_decoder.norm.weight", C); add("complex_decoder.norm.bias", C);
        add("complex_decoder.conv.weight", 2 * C * 2); add("complex_decoder.conv.bias", 2);
    }
};

const Table& table() {
    static const Table t;
    return t;
}
const std::unordered_map<std::string, long long>& offsets() {
    static const std::unordered_map<std::string, long long> m = [] {
        std::unordered_map<std::string, long long> o;
        for (const Entry& e : table().e) o.emplace(e.key, e.off);
        return o;
    }();
    return m;
}

// ---- one forward pass = a walk over the launch list; `dry` only sizes the workspace
struct Run {
    const float* P;             // parameter block (null in a dry run)
    char* ws;                   // workspace base
    size_t top = 0, peak = 0, cap = 0;
    bool dry;
    int precision;
    cudaStream_t st;
    const int* frames = nullptr;    // ragged batch: valid frames per batch item (device), null = every item has all T frames
    int T = 0;
    int rc = 0;

    const float* w(const std::string& key) const {
        if (dry) return nullptr;
        const auto it = offsets().find(key);
        if (it != offsets().end()) return P + it->second;
        cmgan_set_error("cmgan_tscnet_fwd: unknown parameter %s", key.c_str());
        const_cast<Run*>(this)->rc = -1;
        return nullptr;
    }
    template <typename T = float>
    T* alloc(size_t n) {
        top = (top + 255) & ~(size_t)255;
        T* p = dry ? nullptr : reinterpret_cast<T*>(ws + top);
        top += n * sizeof(T);
        if (top > peak) peak = top;
        if (!dry && top > cap && rc == 0) { cmgan_set_error("cmgan_tscnet_fwd: workspace too small (%zu bytes needed so far, %zu given)", top, cap); rc = -1; }
        return p;
    }
    void ok(int r) { if (r != 0 && rc == 0) rc = r; }
    bool live() const { return !dry && rc == 0; }
};

struct Tabs { float *scale, *shift, *mean, *rstd; int width; };
Tabs make_tabs(Run& r, int G, int width) {
    Tabs t;
    t.scale = r.alloc((size_t)G * width); t.shift = r.alloc((size_t)G * width);
    t.mean = r.alloc((size_t)G * width); t.rstd = r.alloc((size_t)G * width);
    t.width = width;
    return t;
}

struct Gemm {
    CmganGemmArgs a;
    Gemm(const float* A, long long lda, const float* W, long long sb_tap, long long sb_k, long long sb_n, const float* bias, float* Cout,
         long long ldc, long long M, int N, int Cin) {
        memset(&a, 0, sizeof(a));
        a.A = A; a.lda = lda; a.B = W; a.sb_tap = sb_tap; a.sb_k = sb_k; a.sb_n = sb_n; a.bias = bias; a.C = Cout; a.ldc = ldc;
        a.M = (int)M; a.N = N; a.Cin = Cin; a.ntaps = 1;
        a.mul_y = a.mul_x = a.div_y = a.div_x = 1;
        a.inv_keep = 1.f; a.pro_inv_keep = 1.f; a.alpha = 1.f; a.pro_alpha = 1.f;
    }
    Gemm& conv(int OH, int OW, int IH, int IW, int mul_x = 1) {
        a.conv = 1; a.OH = OH; a.OW = OW; a.IH = IH; a.IW = IW; a.mul_x = mul_x;
        return *this;
    }
    Gemm& taps(int n, const int* dy, const int* dx) {
        a.ntaps = n;
        for (int i = 0; i < n; ++i) { a.dy[i] = dy[i]; a.dx[i] = dx[i]; }
        return *this;
    }
    Gemm& residual(const float* R, long long ldr) { a.epi = CMGAN_EPI_DROP_RES; a.R = R; a.ldr = ldr; return *this; }
    void run(Run& r) {
        a.precision = r.precision;
        if (r.precision == 1 && a.N % 16 == 0 && a.N <= 256 && a.Cin % 32 == 0) {      // scratch for the re-tiled weight (gemm_args.h)
            a.ws_floats = (long long)a.N * a.Cin * a.ntaps;
            a.ws = r.alloc((size_t)a.ws_floats);
        }
        if (r.live()) r.ok(cmgan_gemm_rows_f32(&a, r.st));
    }
};

void inst_norm_site(Run& r, const float* x, long long ldx, int G, long long rows, int Cn, const float* gamma, const float* beta, const Tabs& t,
                    double*& sums) {
    double* s = sums;
    sums += (size_t)G * Cn * 2;
    if (!r.live()) return;
    if (r.frames) {         // a group's statistics span its valid frames only; rows / T rows per frame (F, F2 or 2 F2 at the sites below)
        r.ok(cmgan_norm_stats_varlen(x, ldx, G, rows, Cn, r.frames, rows / r.T, s, r.st));
        r.ok(cmgan_norm_finalize_varlen(s, r.frames, rows / r.T, r.T, G, Cn, gamma, beta, t.scale, t.shift, t.mean, t.rstd, t.width, r.st));
        return;
    }
    r.ok(cmgan_norm_stats(x, ldx, G, rows, Cn, s, r.st));
    r.ok(cmgan_norm_finalize(s, rows, G, Cn, 0, gamma, beta, nullptr, nullptr, 0.f, t.scale, t.shift, t.mean, t.rstd, t.width, r.st));
}

// InstanceNorm2d(affine) + PReLU of a raw (M, 64) tensor, written into dst (generator.py:35-37)
void norm_prelu_to(Run& r, const float* raw, int G, long long rows, const float* gamma, const float* beta, const float* slope, float* dst,
                   long long ldd, double*& sums) {
    Tabs t = make_tabs(r, G, C);
    inst_norm_site(r, raw, C, G, rows, C, gamma, beta, t, sums);
    if (r.live()) r.ok(cmgan_norm_apply(raw, C, G, rows, C, 1 | (r.precision == 1 ? 16 : 0), t.scale, t.shift, C, slope, dst, ldd, r.st));
}

// DilatedDenseNet (generator.py:39-47) on the concat buffer cat = [out4 | out3 | out2 | out1 | x]
void dense_block(Run& r, float* cat, const std::string& p, int B, int T, int Fw, double*& sums) {
    const long long M = (long long)B * T * Fw, rows = (long long)T * Fw;
    for (int i = 1; i <= 4; ++i) {
        const int dil = 1 << (i - 1), c0 = (5 - i) * C, Cin = C * i, co = (4 - i) * C;
        const std::string s = std::to_string(i);
        float* raw = r.alloc((size_t)M * C);
        const int dy[6] = {-dil, -dil, -dil, 0, 0, 0}, dx[6] = {-1, 0, 1, -1, 0, 1};         // tap = kh * 3 + kw, causal in time (generator.py:12-21)
        Gemm(cat ? cat + c0 : nullptr, CAT, r.w(p + "conv" + s + ".weight"), 1, 6, (long long)Cin * 6, r.w(p + "conv" + s + ".bias"), raw, C, M, C, Cin)
            .taps(6, dy, dx).conv(T, Fw, T, Fw).run(r);
        norm_prelu_to(r, raw, B, rows, r.w(p + "norm" + s + ".weight"), r.w(p + "norm" + s + ".bias"), r.w(p + "prelu" + s + ".weight"),
                      cat ? cat + co : nullptr, CAT, sums);
    }
}

// 0.5 * FF(LN(x)) + x  (conformer.py:54-72,136-148,211-212)
float* feed_forward(Run& r, const float* xin, long long M, const std::string& p) {
    float* out = r.alloc((size_t)M * C);
    if (r.precision == 1) {          // fused kernel: hidden activation in TMEM / shared memory only (ffn_fused.cu)
        float* w1p = r.alloc((size_t)4 * C * C);
        float* w2p = r.alloc((size_t)4 * C * C);
        if (r.live()) {
            r.ok(cmgan_pack_weight(r.w(p + "fn.fn.net.0.weight"), w1p, 0, 1, C, C, 1, 4 * C, r.st));
            r.ok(cmgan_pack_weight(r.w(p + "fn.fn.net.3.weight"), w2p, 0, 1, 4 * C, 4 * C, 1, C, r.st));
            r.ok(cmgan_ffn_fwd(xin, C, M, r.w(p + "fn.norm.weight"), r.w(p + "fn.norm.bias"), w1p, r.w(p + "fn.fn.net.0.bias"), w2p,
                               r.w(p + "fn.fn.net.3.bias"), 0.5f, 0ull, 0ull, 0u, 1.f, nullptr, out, C, r.st));
        }
        return out;
    }
    float* xn = r.alloc((size_t)M * C);
    float* stt = r.alloc((size_t)M * 2);
    float* a = r.alloc((size_t)M * 4 * C);
    if (r.live()) r.ok(cmgan_ln_apply(xin, C, M, r.w(p + "fn.norm.weight"), r.w(p + "fn.norm.bias"), nullptr, 0, xn, C, stt, 0, r.st));
    Gemm g1(xn, C, r.w(p + "fn.fn.net.0.weight"), 0, 1, C, r.w(p + "fn.fn.net.0.bias"), nullptr, 4 * C, M, 4 * C, C);
    g1.a.epi = CMGAN_EPI_SWISH_DUAL; g1.a.C2 = a; g1.a.ldc2 = 4 * C;
    g1.run(r);
    Gemm g2(a, 4 * C, r.w(p + "fn.fn.net.3.weight"), 0, 1, 4 * C, r.w(p + "fn.fn.net.3.bias"), out, C, M, C, 4 * C);
    g2.residual(xin, C).a.alpha = 0.5f;
    g2.run(r);
    return out;
}

// ConformerBlock + the outer TSCB residual (conformer.py:216-222, generator.py:95,97): returns LN(x4) + x in `y`
void conformer(Run& r, const float* x, float* y, const std::string& p, int B, int T, int F2, int axis) {
    const long long M = (long long)B * T * F2;
    const size_t mark = r.top;
    const int rnd = r.precision == 1 ? 1 : 0;
    float* x1 = feed_forward(r, x, M, p + "ff1.");
    // ---- attention (conformer.py:90-133)
    float* xn2 = r.alloc((size_t)M * C);
    float* st2 = r.alloc((size_t)M * 2);
    if (r.live()) r.ok(cmgan_ln_apply(x1, C, M, r.w(p + "attn.norm.weight"), r.w(p + "attn.norm.bias"), nullptr, 0, xn2, C, st2, rnd, r.st));
    float* qkv = r.alloc((size_t)M * 3 * C);
    // to_q and to_kv are adjacent in the parameter block: one (192, 64) projection
    Gemm(xn2, C, r.w(p + "attn.fn.to_q.weight"), 0, 1, C, nullptr, qkv, 3 * C, M, 3 * C, C).run(r);
    float* ctx = r.alloc((size_t)M * C);
    float* lse = r.alloc((size_t)M * 4);
    if (r.live()) {
        const float* E = r.w(p + "attn.fn.rel_pos_emb.weight");
        if (r.frames)
            r.ok(r.precision == 1 ? cmgan_attention_fwd_tf32_varlen(qkv, E, B, T, F2, axis, r.frames, ctx, lse, r.st)
                                  : cmgan_attention_fwd_varlen(qkv, E, B, T, F2, axis, r.frames, ctx, lse, r.st));
        else
            r.ok(r.precision == 1 ? cmgan_attention_fwd_tf32(qkv, E, B, T, F2, axis, ctx, lse, r.st) : cmgan_attention_fwd(qkv, E, B, T, F2, axis, ctx, lse, r.st));
    }
    float* x2 = r.alloc((size_t)M * C);
    Gemm(ctx, C, r.w(p + "attn.fn.to_out.weight"), 0, 1, C, r.w(p + "attn.fn.to_out.bias"), x2, C, M, C, C).residual(x1, C).run(r);
    // ---- convolution module (conformer.py:160-173)
    float* xn3 = r.alloc((size_t)M * C);
    float* st3 = r.alloc((size_t)M * 2);
    if (r.live()) r.ok(cmgan_ln_apply(x2, C, M, r.w(p + "conv.net.0.weight"), r.w(p + "conv.net.0.bias"), nullptr, 0, xn3, C, st3, rnd, r.st));
    float* g = r.alloc((size_t)M * 4 * C);
    Gemm(xn3, C, r.w(p + "conv.net.2.weight"), 0, 1, C, r.w(p + "conv.net.2.bias"), g, 4 * C, M, 4 * C, C).run(r);
    float* d = r.alloc((size_t)M * 2 * C);
    Tabs bn = make_tabs(r, 1, 2 * C);
    float* dsw = r.alloc((size_t)M * 2 * C);
    if (r.live()) {
        if (r.frames)
            r.ok(cmgan_glu_dwconv_fwd_varlen(g, r.w(p + "conv.net.4.conv.weight"), r.w(p + "conv.net.4.conv.bias"), B, T, F2, axis, r.frames, d, r.st));
        else
            r.ok(cmgan_glu_dwconv_fwd(g, r.w(p + "conv.net.4.conv.weight"), r.w(p + "conv.net.4.conv.bias"), B, T, F2, axis, d, nullptr, r.st));
        // eval: BatchNorm1d folds to scale / shift from the running statistics (mode 1; they are only read)
        r.ok(cmgan_norm_finalize(nullptr, M, 1, 2 * C, 1, r.w(p + "conv.net.5.weight"), r.w(p + "conv.net.5.bias"),
                                 const_cast<float*>(r.w(p + "conv.net.5.running_mean")), const_cast<float*>(r.w(p + "conv.net.5.running_var")), 0.1f,
                                 bn.scale, bn.shift, bn.mean, bn.rstd, 2 * C, r.st));
        r.ok(cmgan_norm_apply(d, 2 * C, 1, M, 2 * C, 2 | (16 * rnd), bn.scale, bn.shift, 2 * C, nullptr, dsw, 2 * C, r.st));
    }
    float* x3 = r.alloc((size_t)M * C);
    Gemm(dsw, 2 * C, r.w(p + "conv.net.7.weight"), 0, 1, 2 * C, r.w(p + "conv.net.7.bias"), x3, C, M, C, 2 * C).residual(x2, C).run(r);
    // ---- second feed-forward, post norm, outer residual
    float* x4 = feed_forward(r, x3, M, p + "ff2.");
    float* st5 = r.alloc((size_t)M * 2);
    if (r.live()) r.ok(cmgan_ln_apply(x4, C, M, r.w(p + "post_norm.weight"), r.w(p + "post_norm.bias"), x, C, y, C, st5, 0, r.st));
    r.top = mark;            // everything but `y` (owned by the caller) is released
}

void forward(Run& r, const float* x, long long sxb, long long sxc, long long sxt, long long sxf, int B, int T, int F, float* fr, float* fi) {
    const int F2 = (F - 1) / 2 + 1;
    const long long M = (long long)B * T * F, M2 = (long long)B * T * F2;
    const size_t n_sums = (size_t)(16 * C + 2) * B * 2 + 64;
    double* sums0 = r.alloc<double>(n_sums);
    double* sums = sums0;
    if (r.live()) {
        cudaError_t e = cudaMemsetAsync(sums0, 0, n_sums * sizeof(double), r.st);
        if (e != cudaSuccess) { cmgan_set_error("cmgan_tscnet_fwd: cudaMemsetAsync: %s", cudaGetErrorString(e)); r.rc = -1; }
    }
    float* hA = r.alloc((size_t)M2 * C);          // TSCB activations ping-pong between these two
    float* hB = r.alloc((size_t)M2 * C);
    // ---- dense encoder (generator.py:50-69)
    {
        const size_t mark = r.top;
        const std::string pe = "dense_encoder.";
        float* catE = r.alloc((size_t)M * CAT);
        float* raw0 = r.alloc((size_t)M * C);
        if (r.live()) r.ok(cmgan_head_conv(x, sxb, sxc, sxt, sxf, B, T, F, r.w(pe + "conv_1.0.weight"), r.w(pe + "conv_1.0.bias"), raw0, C, r.st));
        norm_prelu_to(r, raw0, B, (long long)T * F, r.w(pe + "conv_1.1.weight"), r.w(pe + "conv_1.1.bias"), r.w(pe + "conv_1.2.weight"),
                      catE ? catE + 4 * C : nullptr, CAT, sums);
        dense_block(r, catE, pe + "dilated_dense.", B, T, F, sums);
        float* e2 = r.alloc((size_t)M2 * C);
        const int dy[3] = {0, 0, 0}, dx[3] = {-1, 0, 1};
        Gemm(catE, CAT, r.w(pe + "conv_2.0.weight"), 1, 3, 3 * C, r.w(pe + "conv_2.0.bias"), e2, C, M2, C, C).taps(3, dy, dx).conv(T, F2, T, F, 2).run(r);
        Tabs t2 = make_tabs(r, B, C);
        inst_norm_site(r, e2, C, B, (long long)T * F2, C, r.w(pe + "conv_2.1.weight"), r.w(pe + "conv_2.1.bias"), t2, sums);
        if (r.live()) r.ok(cmgan_norm_apply(e2, C, B, (long long)T * F2, C, 1, t2.scale, t2.shift, C, r.w(pe + "conv_2.2.weight"), hA, C, r.st));
        r.top = mark;
    }
    // ---- 4 x TSCB (generator.py:92-99): time conformer then frequency conformer on the same rows
    float *h = hA, *hn = hB;
    for (int i = 1; i <= 4; ++i)
        for (int axis = 0; axis < 2; ++axis) {
            conformer(r, h, hn, "TSCB_" + std::to_string(i) + (axis == 0 ? ".time_conformer." : ".freq_conformer."), B, T, F2, axis);
            float* t = h; h = hn; hn = t;
        }
    // ---- decoders (generator.py:122-156)
    float* sp[2];
    const char* names[2] = {"mask_decoder.", "complex_decoder."};
    for (int dd = 0; dd < 2; ++dd) {
        const std::string pd = names[dd];
        sp[dd] = r.alloc((size_t)M2 * 2 * C);          // (B, T, 2 F2, 64): the sub-pixel shuffle is a reinterpretation
        const size_t mark = r.top;
        float* cat = r.alloc((size_t)M2 * CAT);
        if (r.live()) r.ok(cmgan_copy_rows_operand(h, C, cat + 4 * C, CAT, M2, C, r.st));
        dense_block(r, cat, pd + "dense_block.", B, T, F2, sums);
        const int dy[3] = {0, 0, 0}, dx[3] = {-1, 0, 1};
        Gemm(cat, CAT, r.w(pd + "sub_pixel.conv.weight"), 1, 3, 3 * C, r.w(pd + "sub_pixel.conv.bias"), sp[dd], 2 * C, M2, 2 * C, C)
            .taps(3, dy, dx).conv(T, F2, T, F2).run(r);
        r.top = mark;
    }
    const std::string pm = "mask_decoder.", pc = "complex_decoder.";
    float* m1 = r.alloc((size_t)M);
    Tabs tabM = make_tabs(r, B, 1), tabC = make_tabs(r, B, C);
    float* cplx = r.alloc((size_t)M * 2);
    if (r.live()) r.ok(cmgan_rowdot_fwd(sp[0], B, T, F, 1, nullptr, nullptr, nullptr, r.w(pm + "conv_1.weight"), r.w(pm + "conv_1.bias"), m1, r.st));
    inst_norm_site(r, m1, 1, B, (long long)T * F, 1, r.w(pm + "norm.weight"), r.w(pm + "norm.bias"), tabM, sums);
    inst_norm_site(r, sp[1], C, B, (long long)T * 2 * F2, C, r.w(pc + "norm.weight"), r.w(pc + "norm.bias"), tabC, sums);
    if (r.live()) {
        r.ok(cmgan_rowdot_fwd(sp[1], B, T, F, 2, tabC.scale, tabC.shift, r.w(pc + "prelu.weight"), r.w(pc + "conv.weight"), r.w(pc + "conv.bias"), cplx, r.st));
        r.ok(cmgan_recombine(m1, tabM.scale, tabM.shift, r.w(pm + "prelu.weight"), r.w(pm + "final_conv.weight"), r.w(pm + "final_conv.bias"),
                             r.w(pm + "prelu_out.weight"), x, sxb, sxc, sxt, sxf, cplx, B, T, F, fr, fi, r.st));
    }
    if ((size_t)(sums - sums0) > n_sums && r.rc == 0) { cmgan_set_error("cmgan_tscnet_fwd: statistics scratch exhausted"); r.rc = -1; }
}

}  // namespace

CMGAN_API int cmgan_tscnet_param_count(void) { return (int)table().e.size(); }
CMGAN_API long long cmgan_tscnet_param_floats(void) { return table().total; }

CMGAN_API int cmgan_tscnet_param_info(int index, const char** key, long long* offset, long long* numel) {
    CMGAN_REQUIRE(index >= 0 && index < (int)table().e.size(), "cmgan_tscnet_param_info: index %d out of range", index);
    const Entry& e = table().e[index];
    if (key) *key = e.key.c_str();
    if (offset) *offset = e.off;
    if (numel) *numel = e.numel;
    return 0;
}

CMGAN_API long long cmgan_tscnet_workspace_bytes(int B, int T, int F, int precision) {
    if (B <= 0 || T <= 0 || F != NFEAT || (precision != 0 && precision != 1)) { cmgan_set_error("cmgan_tscnet_workspace_bytes: bad arguments"); return -1; }
    Run r;
    r.P = nullptr; r.ws = nullptr; r.dry = true; r.precision = precision; r.st = nullptr;
    forward(r, nullptr, 0, 0, 0, 0, B, T, F, nullptr, nullptr);
    return (long long)r.peak + 256;
}

// Ragged batch (inference on clips of different lengths in one pass): frames = device int[B], 1 <= frames[b] <= T.  For t < frames[b] the
// outputs equal cmgan_tscnet_fwd on x[b, :, :frames[b]] alone; rows t >= frames[b] of x are never read by a valid row (the convolutions
// are causal in time; attention, the depthwise convolution and the InstanceNorm statistics stop at frames[b]) and their outputs are
// unspecified.  frames == NULL is cmgan_tscnet_fwd.  The workspace is the one cmgan_tscnet_workspace_bytes(B, T, F, precision) gives.
CMGAN_API int cmgan_tscnet_fwd_varlen(const float* params, const float* x, long long sxb, long long sxc, long long sxt, long long sxf, int B, int T,
                                      int F, const int* frames, float* final_real, float* final_imag, void* workspace, long long workspace_bytes,
                                      int precision, void* stream) {
    CMGAN_REQUIRE(params && x && final_real && final_imag && workspace, "cmgan_tscnet_fwd: null pointer");
    CMGAN_REQUIRE(B > 0 && T > 0 && F == NFEAT, "cmgan_tscnet_fwd: expected x of shape (B, 2, T, %d), got B=%d T=%d F=%d", NFEAT, B, T, F);
    CMGAN_REQUIRE(precision == 0 || precision == 1, "cmgan_tscnet_fwd: precision must be 0 (fp32) or 1 (tf32)");
    CMGAN_REQUIRE((((uintptr_t)params) & 15) == 0 && (((uintptr_t)workspace) & 255) == 0, "cmgan_tscnet_fwd: params must be 16-byte, workspace 256-byte aligned");
    cmgan_set_tf32_rounding(precision);       // producers of tensor-core operands round to nearest on store (library-wide switch)
    Run r;
    r.P = params; r.ws = static_cast<char*>(workspace); r.cap = (size_t)workspace_bytes; r.dry = false; r.precision = precision;
    r.st = (cudaStream_t)stream;
    r.frames = frames; r.T = T;
    forward(r, x, sxb, sxc, sxt, sxf, B, T, F, final_real, final_imag);
    return r.rc;
}

CMGAN_API int cmgan_tscnet_fwd(const float* params, const float* x, long long sxb, long long sxc, long long sxt, long long sxf, int B, int T, int F,
                               float* final_real, float* final_imag, void* workspace, long long workspace_bytes, int precision, void* stream) {
    return cmgan_tscnet_fwd_varlen(params, x, sxb, sxc, sxt, sxf, B, T, F, nullptr, final_real, final_imag, workspace, workspace_bytes, precision,
                                   stream);
}
